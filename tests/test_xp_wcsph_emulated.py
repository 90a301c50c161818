"""The WCSPH step per particle against the extended-precision restatement of tests/xp_wcsph.py, in
strict and fast arithmetic, on the CPU: the oracle's strict closures and the FAST_MATH closures of
csrc/wcsph_ops.cuh run by the emulation harness (tests/emu/emu_pairs.cpp, `rsqrt` = 1/sqrt).

Both passes start from the same FP64 inputs on both sides: the density pass from the post-drift
x, h, m the harness is given, the force pass and kick from the harness's own rho, rho', h, P, P'
and the given half-step v.  The given v has the mean fluid velocity removed: the kick's increment
0.5 dt Dv is then resolved in v instead of lost below an ulp of the mean flow.

Two gates, with u = 2^-53 and scale the error scale of xp_wcsph (a magnitude bound per term,
summed over the accepted pairs, propagated through the per-particle formulas):

* rigorous, per particle:  |y - y_xp| <= (n + C) u scale, with n = n_p for the density outputs and
  2 n_p for v.  A pair term of either arithmetic is a fixed chain of at most ~24 FP64 operations
  (dx: 1, r^2: 3 or 5, sqrt or rsqrt + Newton: 2, x = r/h: 1, the kernel polynomial and its
  constant: 6 to 8, the pressure and viscosity factors: 8), each with a relative error of at most
  u, and libdevice's rsqrt 1 ulp, sqrt and division 0 in the default build; the error scale of the
  term already carries the magnitudes of every operand that can cancel and the condition with
  respect to r (|x dW/dx|).  Recursive summation of n terms adds at most gamma_n ~ n u of the sum
  of magnitudes; the strict force pass adds the pressure and the viscous term separately (2 per
  pair), the fast one with one FMA.  The per-particle finish adds exp (1 ulp) of an argument
  with 3 roundings (counted by its |arg| in the scale), sqrt or cbrt (1 ulp), a subtraction, the
  pressure's 4 operations and the kick's 6.  C = 32 covers these with room.
* statistical, per output field: the median and the 99th percentile of |y - y_xp| / (u scale)
  stay below the thresholds of GATES.  These are what would catch a constant wrong in its 14th
  digit or a square root seeded in single precision, which the rigorous gate is too wide for.
"""
import subprocess

import numpy as np
import pytest

import xp_wcsph as X
from sph_mountain_waves_b200 import cases
from test_emulated_kernels import CASES, CSRC, EMU, ROOT, advanced_state, finish_step, run_emulation
from test_oracle_vs_numpy_closures import numpy_step_kick_drift, numpy_step_sums
from util import load_oracle, rel_err

C_OPS = 32
# (median, 99th percentile) ceilings of err / (u scale).  Measured on the emulation (x86-64, glibc,
# -ffp-contract=off) over hill3d, witch2d, long3d, long2d, strict and fast, both strides and cell
# orders; the worst case over all of them is in the comment.  Margin: about 2x the worst median and
# 1.5x the worst 99th percentile, kept below what the mutations listed in DESIGN.md §2 give.
GATES = {
    "rho":   (1.0, 3.0),     # measured <= 0.51 / 1.66   (cw +1e-14: 18 / 25)
    "rho_p": (0.8, 2.5),     # measured <= 0.33 / 1.14
    "h":     (0.6, 2.0),     # measured <= 0.22 / 0.78
    "P":     (0.4, 1.5),     # measured <= 0.10 / 0.58
    "v":     (0.6, 2.0),     # measured <= 0.25 / 1.10   (force constant +1e-14: 1.62 / 2.58)
}


@pytest.fixture(scope="session")
def emu_pairs_binary():
    out = EMU / "build" / "emu_pairs"
    out.parent.mkdir(exist_ok=True)
    deps = [EMU / "emu_pairs.cpp", EMU / "cuda_runtime.h"] + sorted(CSRC.glob("*.cuh")) + \
           [CSRC / "sphmw_internal.h", CSRC / "grid_setup.cpp"]
    if not out.exists() or any(d.stat().st_mtime > out.stat().st_mtime for d in deps):
        subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-Wno-attributes", "-DSPHMW_EMU",
                        f"-I{EMU}", f"-I{ROOT / 'include'}", f"-I{CSRC}", str(EMU / "emu_pairs.cpp"),
                        str(CSRC / "grid_setup.cpp"), "-o", str(out)], check=True)
    return out


def without_mean_flow(fields, p):
    f = dict(fields)
    fluid = f["type"] == p["fluid"]
    f["v"] = f["v"] - fluid[:, None] * f["v"][fluid].mean(axis=0)[None, :]
    return f


def gate(label, field, dev, ref, scale, K, gates=GATES):
    """both gates for one output field; returns (p50, p99, max) of the ratio"""
    rat, bad = X.ratios(dev, ref, scale)
    assert bad == 0, f"{label} {field}: {bad} non-finite values of the wrong class"
    K = np.broadcast_to(np.asarray(K, dtype=np.float64).reshape(K.shape[0], *([1] * (np.ndim(dev) - 1))), np.shape(dev))
    fin = np.isfinite(np.asarray(ref, dtype=X.LD))
    over = rat > K[fin] + C_OPS
    assert not over.any(), f"{label} {field}: rigorous bound broken at {int(over.sum())} values, worst ratio {float(rat.max()):.3g}"
    r = rat.astype(np.float64)
    p50, p99 = (float(np.percentile(r, q)) for q in (50, 99)) if r.size else (0.0, 0.0)
    lim50, lim99 = gates[field]
    assert p50 <= lim50 and p99 <= lim99, f"{label} {field}: median {p50:.3g} (<= {lim50}), p99 {p99:.3g} (<= {lim99})"
    return p50, p99, float(r.max()) if r.size else 0.0


def check_passes(label, case, fields, got, n_pairs):
    """the density pass against xp on the given x, h, m; the force pass + kick against xp on the
    given x, v and the device's rho, rho', h, P, P'"""
    dim, p = case.dim, case.params
    den = X.density(fields, p, case.h, dim)
    assert int(den["n_p"].sum()) == n_pairs
    for f, s in (("rho", "s_rho"), ("rho_p", "s_rho_p"), ("h", "s_h"), ("P", "s_P")):
        gate(label, f, got[f], den[f], den[s], den["n_p"])
    fin = dict(fields, h=got["h"], rho=got["rho"], rho_p=got["rho_p"], P=got["P"], P_p=got["P_p"])
    fk = X.force_kick(fin, p, case.h, dim)
    fluid = fields["type"] == p["fluid"]
    assert np.array_equal(got["v"][~fluid], fields["v"][~fluid])   # walls and mountain keep v
    gate(label, "v", got["v"][fluid, :dim], fk["v"][fluid, :dim], fk["s_v"][fluid, :dim], 2 * fk["n_p"][fluid])


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("fast,stride,cx_shift", [(0, 40, -1), (1, 40, -1), (1, 8, -1), (1, 40, 2)],
                         ids=["strict", "fast", "fast-overflow", "fast-xchunk"])
def test_emulated_step_against_extended_precision(emu_pairs_binary, tmp_path, name, fast, stride, cx_shift):
    """strict: the oracle's arithmetic (the emulated strict closures equal it bit for bit,
    test_emulated_kernels.py); fast: the FAST_MATH closures, also on every particle's overflow
    path (stride 8 walks the cells) and on the x-chunked cell order"""
    case = CASES[name]()
    _, fields = advanced_state(case)
    fields = without_mean_flow(fields, case.params)
    meta, got = run_emulation(emu_pairs_binary, tmp_path, case, fields, fast=fast, stride=stride, cx_shift=cx_shift)
    assert (meta["overflow"] > 0) == (stride == 8)
    check_passes(f"{name} fast={fast} stride={stride}", case, fields, got, meta["pairs_density"])


def test_oracle_step_against_extended_precision():
    """the oracle's own operator sequence, staged the same way"""
    case = CASES["hill3d"]()
    o, fields = advanced_state(case)
    pairs = finish_step(o)
    got = {f: o.field(f) for f in ("rho", "rho_p", "h", "P", "P_p", "v")}
    # the kick started from the oracle's v after move!, which `fields` holds
    check_passes("oracle", case, fields, got, pairs)


def test_kick_and_drift_against_extended_precision():
    case = CASES["witch2d"]()
    o = load_oracle(case)
    o.create_cell_list()
    o.step("wcsph", 2)
    state = {k: o.field(k) for k in ("x", "v", "rho", "rho_p", "type")}
    o.apply("wcsph.accelerate")
    v_half = o.field("v")
    o.apply("wcsph.move")
    kd = X.kick_drift(state, case.params)
    n = np.zeros(case.n, dtype=np.int64)
    gates = {"v": (0.6, 2.0), "x": (0.6, 2.0)}
    gate("kick", "v", v_half, kd["v"], kd["s_v"], n, gates)
    gate("drift", "x", o.field("x"), kd["x"], kd["s_x"], n, gates)


# ---------------------------------------------------------------------------------------------
# the reference itself
# ---------------------------------------------------------------------------------------------
def perturbed(case, seed):
    rng = np.random.default_rng(seed)
    fluid = case.fields["type"] == 0.0
    case.fields["v"] = case.fields["v"] + fluid[:, None] * rng.normal(scale=8.0, size=(case.n, 3)) * \
        np.array([1.0, 1.0, 1.0 if case.dim == 3 else 0.0])
    case.fields["h"] = case.fields["h"] * rng.uniform(0.9, 1.3, case.n)
    return case


@pytest.mark.parametrize("make", [
    lambda: cases.mountain_wave_2d(n_y=12.0, dom_length=30e3, h_m=3000.0, a=6e3, U=25.0),
    lambda: cases.bell_hill_3d(10, 8, 6, h_m=3000.0, a=4e3, U=25.0),
])
def test_xp_agrees_with_the_fp64_restatement(make):
    """xp's three stages, chained through FP64, against numpy_step_sums (a different summation
    order and FP64 throughout): to 1e-12"""
    case = perturbed(make(), 11)
    f = {k: v.copy() for k, v in case.fields.items()}
    numpy_step_kick_drift(f, case.params)
    kd = X.kick_drift(case.fields, case.params)
    assert rel_err(kd["v"].astype(np.float64), f["v"]) < 1e-12
    assert rel_err(kd["x"].astype(np.float64), f["x"]) < 1e-12
    staged = dict(case.fields, x=kd["x"].astype(np.float64), v=kd["v"].astype(np.float64))
    npairs = numpy_step_sums(f, case.params, case.h, case.dim == 3)
    den = X.density(staged, case.params, case.h, case.dim)
    assert int(den["n_p"].sum()) == npairs
    got = {k: den[k].astype(np.float64) for k in ("rho", "rho_p", "h", "P", "P_p")}
    for k in ("rho", "rho_p", "h", "P", "P_p"):
        assert rel_err(got[k], f[k]) < 1e-12, k
    fk = X.force_kick(dict(staged, **got), case.params, case.h, case.dim)
    assert rel_err(fk["v"].astype(np.float64), f["v"]) < 1e-12


def test_xp_agrees_with_mpmath_at_40_digits():
    """rho and Dv of 40 sampled particles of a 3D case, evaluated pair by pair in mpmath at 40
    digits from the same FP64 inputs: to 1e-17 of the error scale"""
    mpmath = pytest.importorskip("mpmath", reason="mpmath (a torch dependency) is needed for the 40-digit check")
    mp = mpmath.mp
    mp.dps = 40
    case = perturbed(cases.bell_hill_3d(10, 8, 6, h_m=3000.0, a=4e3, U=25.0), 12)
    p = case.params
    f = {k: v.copy() for k, v in case.fields.items()}
    numpy_step_kick_drift(f, p)
    numpy_step_sums(f, p, case.h, True)      # gives FP64 rho, rho', P, P', h to stage the force pass from
    sample = np.random.default_rng(1).choice(np.nonzero(f["type"] == 0.0)[0], 40, replace=False)
    den = X.density(f, p, case.h, 3, targets=sample)
    fk = X.force_kick(f, p, case.h, 3, targets=sample)
    i, j = X.neighbour_pairs(f["x"], case.h, sample)
    M = lambda a: mpmath.mpf(float(a))   # noqa: E731
    pi = mpmath.pi
    for s in sample:
        js = j[i == s]
        rho = mpmath.mpf(0)
        Dv = [mpmath.mpf(0)] * 3
        xs = [M(f["x"][s, k]) for k in range(3)]
        rfl = lambda q: max(M(f["rho"][q]), M(p["rho_floor"]))                  # noqa: E731
        pr2 = lambda q: M(f["P_p"][q]) / rfl(q) ** 2                             # noqa: E731
        cs = lambda q: mpmath.sqrt(M(p["gamma"]) * M(f["P"][q]) / rfl(q))      # noqa: E731
        for q in js:
            d = [xs[k] - M(f["x"][q, k]) for k in range(3)]
            r = mpmath.sqrt(d[0] ** 2 + d[1] ** 2 + d[2] ** 2)
            x = r / M(f["h"][s])
            if x <= 1:
                rho += M(f["m"][q]) * 21 / (2 * pi) * (1 - x) ** 4 * (1 + 4 * x) / M(f["h"][s]) ** 3
            hij = (M(f["h"][s]) + M(f["h"][q])) / 2
            x = r / hij
            ker = -210 / pi * (1 - x) ** 3 / hij ** 5 if x <= 1 else mpmath.mpf(0)
            dot = sum(d[k] * (M(f["v"][s, k]) - M(f["v"][q, k])) for k in range(3))
            fc = -M(f["m"][q]) * (pr2(s) + pr2(q)) * ker
            if dot < 0:
                mu = hij * dot / (r * r + M(p["eps"]) * hij * hij)
                pij = (-M(p["alpha"]) * (cs(s) + cs(q)) / 2 * mu + M(p["beta"]) * mu * mu) / ((rfl(s) + rfl(q)) / 2)
                fc += -M(f["m"][q]) * pij * ker
            Dv = [Dv[k] + fc * d[k] for k in range(3)]
        assert abs(mpmath.mpf(str(den["rho"][s])) - rho) <= 1e-17 * mpmath.mpf(str(den["s_rho"][s]))
        for k in range(3):
            assert abs(mpmath.mpf(str(fk["Dv"][s, k])) - Dv[k]) <= 1e-17 * mpmath.mpf(str(fk["s_Dv"][s, k])), k

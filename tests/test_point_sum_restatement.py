"""The CPU restatement of the point sum (tests/c/point_sum_oracle.c, the checker of the device) against an
independent brute force in numpy: every particle within h of the point, no cell list.  `count` matches exactly; the other ops to 1e-13 relative,
because the brute force adds the terms in another order."""
import numpy as np
import pytest

import point_cases as pc
import point_oracle

WENDLAND = {2: (2.228169203286535, 2), 3: (3.3422538049298023, 3)}  # kernels.jl:108-115, :156-163


def brute_force(case, pts, ops):
    f = case.fields
    x, m, rho, h = f["x"], f["m"], f["rho"], case.h
    c, p = WENDLAND[case.dim]
    out = np.full((len(ops), len(pts)), np.nan)
    lo, hi = np.array(case.box_min), np.array(case.box_max)
    for i, q in enumerate(pts):
        if not (np.all(lo <= q) and np.all(q <= hi)):
            continue
        d = q - x
        r = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
        a = r <= h
        s = r[a] / h
        W = c * (1.0 - s) ** 4 * (1.0 + 4.0 * s) / h ** p
        for k, op in enumerate(ops):
            base, _, name = op.partition("*")
            if base == "count":
                out[k, i] = float(a.sum())
                continue
            w = m[a] if base == "mW" else m[a] / rho[a]
            if name:
                fld, _, comp = name.partition("[")
                fld = point_oracle.JULIA.get(fld, fld)
                w = w * (f[fld][a, int(comp[0])] if comp else f[fld][a])
            out[k, i] = np.sum(w * W)
    return out


# Grids at least three cells wide on every axis: on narrower ones the reference's linear key wrap visits
# some cells twice (key_diff -1 and +1 - Lx coincide when Lx = 2), which a brute force does not restate.
@pytest.mark.parametrize("make", [pc.hex_2d, pc.witch_2d, pc.hill_3d], ids=["hex2d", "witch2d", "cubic3d"])
def test_point_sum_restatement_equals_brute_force(make):
    case = make()
    ops = pc.ops_for(case)
    pts = pc.sample_points(case, n_random=200)
    got = point_oracle.for_case(case, pts, ops)
    want = brute_force(case, pts, ops)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want[0])
    assert np.array_equal(got[0][ok], want[0][ok])
    assert (want[0][ok] > 0).sum() > ok.sum() // 2
    for k in range(1, len(ops)):
        scale = np.max(np.abs(want[k][ok]))
        if scale == 0.0:  # a field at rest (the hexagonal lattice carries no perturbation)
            assert np.all(got[k][ok] == 0.0), ops[k]
            continue
        err = np.abs(got[k][ok] - want[k][ok]) / np.maximum(np.abs(want[k][ok]), 1e-3 * scale)
        assert err.max() <= 1e-13, ops[k]

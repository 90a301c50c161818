"""The point-sum kernels (csrc/point_sum.cuh: k_point_keys, the sort by home cell, k_point_sum) compiled
for the HOST and run one thread at a time (tests/emu/emu_point_sum.cpp), against the CPU restatement of the
point sum (tests/c/point_sum_oracle.c) with == for every op — no GPU needed.  Both physical cell orders, a 2D hexagonal and a 3D
cubic lattice and a grid two cells wide in x, where the linear key wrap adds cells."""
import struct
import subprocess
from pathlib import Path

import numpy as np
import pytest

import point_cases as pc
import point_oracle
from util import n_mismatch

ROOT = Path(__file__).resolve().parent.parent
EMU = ROOT / "tests" / "emu"
CSRC = ROOT / "sph_mountain_waves_b200" / "csrc"
KIND = {"count": 0, "mW": 1, "VW": 3}
EXTRA = {"v[0]": 0, "v[1]": 1, "v[2]": 2, "rho_p": 3}


@pytest.fixture(scope="session")
def emu_point_binary():
    out = EMU / "build" / "emu_point_sum"
    out.parent.mkdir(exist_ok=True)
    deps = [EMU / "emu_point_sum.cpp", EMU / "cuda_runtime.h", CSRC / "point_sum.cuh", CSRC / "kernels_sph.cuh",
            CSRC / "sphmw_internal.h", CSRC / "grid_setup.cpp", ROOT / "include" / "sphmw.h"]
    if not out.exists() or any(d.stat().st_mtime > out.stat().st_mtime for d in deps):
        subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-Wno-attributes", "-DSPHMW_EMU",
                        f"-I{EMU}", f"-I{ROOT / 'include'}", f"-I{CSRC}", str(EMU / "emu_point_sum.cpp"),
                        str(CSRC / "grid_setup.cpp"), "-o", str(out)], check=True)
    return out


def decode(op):
    base, _, f = op.partition("*")
    return (KIND[base] + (1 if f else 0), EXTRA[point_oracle.JULIA.get(f, f)] if f else -1)


def run_emulation(binary, tmp_path, case, zrun, ops, points):
    f = case.fields
    n, npts = len(f["m"]), len(points)
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as fp:
        fp.write(struct.pack("<4i", int(zrun), len(ops), len(EXTRA), 0))
        fp.write(struct.pack("<2q", n, npts))
        fp.write(struct.pack("<7d", *case.box_min, *case.box_max, case.h))
        for op in ops:
            fp.write(struct.pack("<2i", *decode(op)))
        cols = [f["x"][:, 0], f["x"][:, 1], f["x"][:, 2], f["m"], f["rho"],
                f["v"][:, 0], f["v"][:, 1], f["v"][:, 2], f["rho_p"]]
        for c in cols:
            fp.write(np.ascontiguousarray(c, dtype="<f8").tobytes())
        fp.write(np.ascontiguousarray(np.asarray(points, dtype=np.float64).T, dtype="<f8").tobytes())
    r = subprocess.run([str(binary), str(inp), str(outp)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr + r.stdout
    return np.frombuffer(outp.read_bytes(), dtype="<f8").reshape(len(ops), npts)


CASES = {"hex2d": pc.hex_2d, "witch2d": pc.witch_2d, "cubic3d": pc.hill_3d,
         "narrow2d": lambda: pc.narrow(2), "narrow3d": lambda: pc.narrow(3)}


@pytest.mark.parametrize("zrun", [1, 0], ids=["zrun", "xchunk"])
@pytest.mark.parametrize("name", list(CASES))
def test_emulated_point_sum_equals_the_restatement(emu_point_binary, tmp_path, name, zrun):
    case = CASES[name]()
    ops = pc.ops_for(case)
    pts = pc.sample_points(case)
    got = run_emulation(emu_point_binary, tmp_path, case, zrun, ops, pts)
    want = point_oracle.for_case(case, pts, ops)
    for k, op in enumerate(ops):
        assert n_mismatch(got[k], want[k]) == 0, op
    # the point sets reach what they are meant to
    outside = np.isnan(want[0])
    assert 4 <= outside.sum() < len(pts) // 2
    assert np.all(np.isnan(got[:, outside]))
    assert (want[0] > 0).sum() > len(pts) // 2


def test_narrow_grid_has_points_exactly_h_away_and_wrapped_cells(emu_point_binary, tmp_path):
    """the narrow lattice is dyadic: points h from a particle are accepted (r == h exactly); with two
    columns the key wrap visits some cells twice (key_diff -1 == +1 - Lx), as it does for particles, so
    some particles are counted twice"""
    case = pc.narrow(2)
    x = case.fields["x"]
    pts = x[:10].copy()
    pts[:, 0] += case.h
    d = pts[:, None, :] - x[None, :, :]
    r = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1] + d[..., 2] * d[..., 2])
    assert np.all((r == case.h).any(axis=1))
    got = run_emulation(emu_point_binary, tmp_path, case, 1, ["count"], pts)
    assert n_mismatch(got, point_oracle.for_case(case, pts, ["count"])) == 0
    within = (r <= case.h).sum(axis=1)
    assert np.all(got[0] >= within) and np.any(got[0] > within)

"""The force pass of the fused WCSPH step over the fluid work list (csrc/pair_list.cuh
k_binary_list_fluid), compiled for the HOST and run one thread at a time (tests/emu/emu_fluid_force.cpp),
against the oracle — no GPU needed.

The harness runs whole multi-step calls as one GPU does: the gather writes the fluid flags, the work list
puts the fluid positions first, the force pass evaluates the pairs of those only and runs init() + finish()
alone for the others, with the next step's accelerate!/move! folded into it on every step but the last.
Walls and the mountain are not fluid, so the lattices below have warps of fluid, of non-fluid and of both
kinds.  Every field must equal the oracle's verlet_step! sequence bit for bit (strict arithmetic), and the
pair count of the last force pass must be the oracle's.
"""
import struct
import subprocess
from pathlib import Path

import numpy as np
import pytest

from sph_mountain_waves_b200 import cases
from util import load_oracle, n_mismatch, rel_err

ROOT = Path(__file__).resolve().parent.parent
EMU = ROOT / "tests" / "emu"
CSRC = ROOT / "sph_mountain_waves_b200" / "csrc"
PARAMS = ["dt", "g", "c", "gamma", "alpha", "beta", "eps", "eta", "rho0", "R_mass", "R_gas", "T_bg", "rho_floor",
          "P_floor", "z_t", "z_b", "gamma_r", "fluid"]


@pytest.fixture(scope="session")
def emu_fluid_binary():
    out = EMU / "build" / "emu_fluid_force"
    out.parent.mkdir(exist_ok=True)
    deps = [EMU / "emu_fluid_force.cpp", EMU / "cuda_runtime.h", CSRC / "pair_list.cuh", CSRC / "wcsph_ops.cuh",
            CSRC / "kernels_sph.cuh", CSRC / "cell_gather.cuh", CSRC / "sphmw_internal.h", CSRC / "grid_setup.cpp",
            CSRC / "q_access.cuh"]
    if not out.exists() or any(d.stat().st_mtime > out.stat().st_mtime for d in deps):
        subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-Wno-attributes", "-DSPHMW_EMU",
                        f"-I{EMU}", f"-I{ROOT / 'include'}", f"-I{CSRC}", str(EMU / "emu_fluid_force.cpp"),
                        str(CSRC / "grid_setup.cpp"), "-o", str(out)], check=True)
    return out


def run_emulation(binary, tmp_path, case, fast, nsteps, calls, stride=40):
    fields = case.fields
    n = len(fields["m"])
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as fp:
        fp.write(struct.pack("<6i", int(fast), int(stride), -1, len(PARAMS), int(nsteps), int(calls)))
        fp.write(struct.pack("<q", n))
        fp.write(struct.pack("<7d", *case.box_min, *case.box_max, case.h))
        for name in PARAMS:
            fp.write(name.encode().ljust(16, b"\0"))
            fp.write(struct.pack("<d", float(case.params.get(name, 0.0))))
        for key in ("x", "v"):
            for k in range(3):
                fp.write(np.ascontiguousarray(fields[key][:, k], dtype="<f8").tobytes())
        for key in ("m", "h", "rho", "rho_p", "type"):
            fp.write(np.ascontiguousarray(fields[key], dtype="<f8").tobytes())
    r = subprocess.run([str(binary), str(inp), str(outp)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr + r.stdout
    raw = outp.read_bytes()
    meta = struct.unpack("<6q", raw[:48])
    arr = np.frombuffer(raw[48:], dtype="<f8").reshape(-1, n)
    return dict(n=meta[0], dim=meta[1], pairs=meta[2], n_fluid=meta[3], warps_nonfluid=meta[4], warps_mixed=meta[5]), \
        {"rho": arr[0], "h": arr[1], "v": arr[2:5].T, "x": arr[5:8].T}


CASES = {
    "hill3d": lambda: cases.bell_hill_3d(24, 12, 10, h_m=3000.0, a=8e3, U=20.0),
    "witch2d": lambda: cases.mountain_wave_2d(n_y=24.0, dom_length=80e3, h_m=3000.0, a=10e3, U=20.0),
}


@pytest.mark.parametrize("name", list(CASES))
def test_fluid_force_calls_equal_the_oracle_bit_for_bit(emu_fluid_binary, tmp_path, name):
    """three calls of four steps each (the advance folded into the force pass of the first three steps
    of every call): x, v, rho, h equal the oracle's twelve verlet_step!s exactly"""
    case = CASES[name]()
    meta, got = run_emulation(emu_fluid_binary, tmp_path, case, fast=0, nsteps=4, calls=3)
    o = load_oracle(case)
    o.create_cell_list()
    o.step("wcsph", 12)
    assert meta["n"] == case.n == len(o)
    assert 0 < meta["n_fluid"] < case.n
    assert meta["warps_nonfluid"] > 0 and meta["warps_mixed"] > 0, meta
    assert meta["n_fluid"] == int(np.sum(o.field("type") == case.params["fluid"]))
    assert meta["pairs"] == o.pair_count() > 0
    for f in ("x", "v", "rho", "h"):
        assert n_mismatch(got[f], o.field(f)) == 0, f


@pytest.mark.parametrize("name", list(CASES))
def test_fast_fluid_force_equals_one_step_calls(emu_fluid_binary, tmp_path, name):
    """FAST_MATH closures: one call of six steps gives the bits of six one-step calls (the folded advance
    and the skipped pairs change nothing), within the north star's tolerance of the oracle"""
    case = CASES[name]()
    meta6, got6 = run_emulation(emu_fluid_binary, tmp_path, case, fast=1, nsteps=6, calls=1)
    meta1, got1 = run_emulation(emu_fluid_binary, tmp_path, case, fast=1, nsteps=1, calls=6)
    o = load_oracle(case)
    o.create_cell_list()
    o.step("wcsph", 6)
    assert meta6["pairs"] == meta1["pairs"] == o.pair_count()
    for f in ("x", "v", "rho", "h"):
        assert n_mismatch(got6[f], got1[f]) == 0, f
        assert rel_err(got6[f], o.field(f)) <= 6e-10, f

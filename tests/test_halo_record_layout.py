"""The x-slab halo record layout (csrc/halo_record.cuh), compiled for the HOST behind
tests/emu/cuda_runtime.h (tests/emu/emu_halo_record.cpp): the base record is row for row the
13-row layout of before, for every scheme's rows 8/9, and the adiabatic flow driver's 17-row record
restores every carried field bit for bit and zeroes what the receiver recomputes.  No GPU needed."""
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
EMU = ROOT / "tests" / "emu"
CSRC = ROOT / "sph_mountain_waves_b200" / "csrc"


def test_halo_record_layout_on_the_host(tmp_path):
    out = tmp_path / "emu_halo_record"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-Wno-attributes", "-DSPHMW_EMU",
                    f"-I{EMU}", f"-I{ROOT / 'include'}", f"-I{CSRC}", str(EMU / "emu_halo_record.cpp"), "-o", str(out)],
                   check=True)
    r = subprocess.run([str(out)], capture_output=True, text=True)
    assert r.returncode == 0 and "HALO_RECORD_OK" in r.stdout, r.stdout + r.stderr


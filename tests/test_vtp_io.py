"""libsphmw's .vtp reader/writer on the host (no GPU): round-tripped like
sph_jl/tests/test_IO.jl:32-60 (scalar / vector fields, exact equality)."""
import numpy as np
import pytest

from sph_mountain_waves_b200 import read_vtp, write_vtp
from sph_mountain_waves_b200._capi import SphmwError


@pytest.mark.parametrize("n", [0, 1, 4095, 4096, 4097, 20000])
def test_write_read_round_trip_exact(tmp_path, n):
    """block boundaries of the zlib stream: 32 KiB blocks = 4096 doubles"""
    rng = np.random.default_rng(n)
    pts = rng.normal(size=(n, 3))
    fields = {"ρ": rng.normal(size=n), "v": rng.normal(size=(n, 3)), "type": rng.integers(0, 3, n).astype(float),
              "weird": np.where(rng.random(n) < 0.1, np.nan, rng.normal(size=n))}
    path = str(tmp_path / "frame.vtp")
    write_vtp(path, pts, fields)
    d = read_vtp(path)
    assert d["Points"].shape == (n, 3) and np.array_equal(d["Points"], pts)
    for k, a in fields.items():
        assert d[k].shape == a.shape
        assert np.array_equal(d[k], a, equal_nan=True), k


def test_reader_errors(tmp_path):
    with pytest.raises(SphmwError):
        read_vtp(str(tmp_path / "missing.vtp"))
    bad = tmp_path / "bad.vtp"
    bad.write_text("<VTKFile type=\"PolyData\"><Piece NumberOfPoints=\"1\"></Piece></VTKFile>")
    with pytest.raises(SphmwError):
        read_vtp(str(bad))


def test_threaded_compression_writes_the_same_bytes(tmp_path, monkeypatch):
    """the zlib blocks of a large frame are compressed by several host threads; the file must
    not depend on how many (blocks are independent streams, written in order)"""
    rng = np.random.default_rng(7)
    n = 300_000
    pts = rng.normal(size=(n, 3)).round(3)
    fields = {"ρ": rng.normal(size=n).round(2), "v": rng.normal(size=(n, 3))}
    blobs = []
    for threads in ("1", "3", "8"):
        monkeypatch.setenv("SPHMW_IO_THREADS", threads)
        path = tmp_path / f"frame_t{threads}.vtp"
        write_vtp(str(path), pts, fields)
        blobs.append(path.read_bytes())
    assert blobs[0] == blobs[1] == blobs[2]
    d = read_vtp(str(tmp_path / "frame_t8.vtp"))
    assert np.array_equal(d["Points"], pts) and np.array_equal(d["v"], fields["v"])

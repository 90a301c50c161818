"""Time of the point sums (sphmw_point_sum) on the bench.py default lattice (bell hill 3D, 64.45 M particles,
strict arithmetic), next to the density pass of the same run.

    python scripts/point_sum_probe.py [--nx 1920 --ny 150 --nz 192] [--warmup 3] [--reps 5]

Sections at mid-z (x-y planes) of 2^16, 2^20 and 2^24 points and 2^20 random points in the box, with the
ops {VW, VW*v[0], VW*v[1], VW*rho_p}; each with device-resident (CUDA tensor) and host (numpy) buffers.
The library's CUDA-event timers give point_keys / point_sort / point_sum per call; a host clock around
each call (which ends in a synchronise) gives the whole call.  Prints one JSON line, with the GPU name and
power limit read in the same run.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from sph_mountain_waves_b200.slabs import SlabRun  # noqa: E402

OPS = ["VW", "VW*v[0]", "VW*v[1]", "VW*rho_p"]
KERNELS = ("point_keys", "point_sort", "point_sum")


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def section(box_lo, box_hi, nx, ny):
    xs = np.linspace(box_lo[0], box_hi[0], nx)
    ys = np.linspace(box_lo[1], box_hi[1], ny)
    X, Y = np.meshgrid(xs, ys, indexing="ij")
    pts = np.empty((nx * ny, 3))
    pts[:, 0], pts[:, 1] = X.ravel(), Y.ravel()
    pts[:, 2] = 0.5 * (box_lo[2] + box_hi[2])
    return pts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=1920)
    ap.add_argument("--ny", type=int, default=150)
    ap.add_argument("--nz", type=int, default=192)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe needs a CUDA device"
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        run = SlabRun.bell_hill_3d(args.nx, args.ny, args.nz, device=0, stream=stream.cuda_stream, device_gen=True)
        run.create_cell_list()
        s = run.sys
        run.step(args.warmup)
        s.timing(True)
        s.timing_reset()
        run.step(2)
        rep = s.timing_report()
        n = len(s)
        dens = rep["wcsph.density_fused"]
        density_ms = dens[0] / dens[1]
        d = s.domain
        lo, hi = (d.x1_min, d.x2_min, d.x3_min), (d.x1_max, d.x2_max, d.x3_max)
        rng = np.random.default_rng(5)
        sets = {"section_2^16": section(lo, hi, 512, 128), "section_2^20": section(lo, hi, 2048, 512),
                "section_2^24": section(lo, hi, 8192, 2048),
                "random_2^20": np.asarray(lo) + rng.random((1 << 20, 3)) * (np.asarray(hi) - np.asarray(lo))}
        results = {}
        for name, pts in sets.items():
            for where in ("device", "host"):
                arg = torch.from_numpy(pts).cuda() if where == "device" else pts
                s.point_sum(arg, OPS)  # warm-up: scratch buffers, sort temporaries
                torch.cuda.synchronize()
                s.timing_reset()
                t0 = time.perf_counter()
                for _ in range(args.reps):
                    s.point_sum(arg, OPS)
                torch.cuda.synchronize()
                wall = (time.perf_counter() - t0) / args.reps * 1e3
                rep = s.timing_report()
                k = {kn: rep[kn][0] / rep[kn][1] for kn in KERNELS if kn in rep}
                results[f"{name}_{where}"] = dict(points=len(pts), call_ms=round(wall, 4),
                                                  **{f"{kn}_ms": round(v, 4) for kn, v in k.items()},
                                                  point_sum_ns_per_point=round(k["point_sum"] / len(pts) * 1e6, 3))
        s.timing(False)
    sec = results["section_2^20_device"]
    gate = 3.0 * density_ms / n * (1 << 20)
    print(json.dumps(dict(gpu=gpu_info(), particles=n, density_ms=round(density_ms, 4),
                          density_ns_per_particle=round(density_ms / n * 1e6, 4),
                          gate_point_sum_ms_2_20=round(gate, 4), gate_met=sec["point_sum_ms"] <= gate,
                          results=results)))


if __name__ == "__main__":
    main()

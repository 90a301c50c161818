#!/usr/bin/env python
"""bench.py — particle-steps/s of the WCSPH mountain-wave hot path on N B200s.

    python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  (CPU arm: the oracle port)
    python bench.py ... --dump-outputs DIR                   (+ the state after the last timed step)

A "step" is one verlet_step! (src/current/wcsph_perturbed_witch.jl:309-332) over the
whole particle set.  Workload: BASELINE.json config 4, the 3D bell-hill mountain wave
with ~64 M lattice-initialised particles in total (strong scaling: the same particle
set is split into x-slabs over the N ranks).  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (which may be read-only)

# 3D: algorithmic bytes per particle of the unfused canonical kernels (SURVEY.md §8d)
BYTES_3D = {"K_A": 117, "K_S": 183, "K_B": 72, "K_C": 113, "step": 485}
BYTES_2D = {"K_A": 85, "K_S": 151, "K_B": 64, "K_C": 89, "step": 389}

WORKLOADS = {
    # name: (nx, ny, nz) fluid cells of the cubic lattice; +6 wall layers on every side
    "bell_hill_3d_64M": (1920, 150, 192),
    "bell_hill_3d_8M": (960, 75, 96),
    "bell_hill_3d_1M": (480, 38, 48),
    # BASELINE config 5 (scaling sweep, large end): ~264 M particles; use --device-gen
    "bell_hill_3d_256M": (3100, 240, 320),
    # BASELINE config 3: 2D Witch of Agnesi, dr = 26 km / 510 (one GPU only)
    "witch_2d_4M": None,
    # BASELINE config 2: 2D isothermal atmosphere at rest (hydrostatic well-balance test), ~244 k particles
    "static_2d_250k": None,
}
CASES_2D = {"witch_2d_4M": "witch_2d", "static_2d_250k": "static_atmosphere_2d"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="bell_hill_3d_64M", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-strict", action="store_true")
    ap.add_argument("--no-overlap", action="store_true",
                    help="slabs: plain halo exchange between the drift and the cell list (no overlap)")
    ap.add_argument("--python-transport", action="store_true",
                    help="slabs: move the halo records with torch.distributed from Python (round-1 path) instead "
                         "of the library's own ncclSend/ncclRecv (csrc/slab_comm.cu)")
    ap.add_argument("--device-gen", action="store_true",
                    help="generate the lattice on the GPU (sphmw_generate_mountain_wave) instead of numpy")
    ap.add_argument("--cpu-sample", default="bell_hill_3d_1M")
    ap.add_argument("--flags", type=int, default=0,
                    help="SPHMW_FLAG_*: 0 strict arithmetic (default: FP64 sums bit-identical to the oracle), "
                         "1 FAST_MATH, 2 CELL_PAIRS, +4 NO_PAIR_LIST (walk the cells in every pass), +16 NO_PRETEST, "
                         "+64 TILES (shared-memory tiles, experimental), +128 NO_PACKED_RECORDS (SoA gathers)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the particle state after the last timed step to DIR/<field>.npy (float64, "
                         "global index order; a fixed sample of large runs), to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md).  The timed region
    of the default run is about half a second, so the samples come from NVML in-process every
    20 ms when pynvml is importable (the same counters nvidia-smi prints); nvidia-smi every 200 ms
    otherwise."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.source = "nvidia-smi"
        self._stop = threading.Event()
        self._t = None

    def _run_nvml(self) -> bool:
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self.index)
            mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
            N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
            N.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        except Exception:
            return False
        self.source = "nvml"
        bits = (N.nvmlClocksThrottleReasonHwSlowdown, N.nvmlClocksThrottleReasonHwThermalSlowdown,
                N.nvmlClocksThrottleReasonSwThermalSlowdown, N.nvmlClocksThrottleReasonSwPowerCap)
        while not self._stop.is_set():
            try:
                sm = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
                r = N.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append([str(sm), str(mx)] + ["Active" if r & b else "Not Active" for b in bits])
            except Exception:
                pass
            self._stop.wait(0.02)
        return True

    def _run(self):
        if self._run_nvml():
            return
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.samples.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4)
                          if len(s) > 2 + i and s[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples), "source": self.source}


# --------------------------------------------------------------------------- CPU arm
def cpu_reference(sample: str, steps: int, warmup: int, min_seconds: float = 10.0):
    """The reference's own CPU implementation cannot run here (100 % Julia, no `julia`
    binary in the image): the CPU arm is the C restatement in oracle/ with OpenMP on
    every host core (kind "port").  A bounded sample of the same workload family:
    `steps` steps, extended up to `min_seconds` of CPU work (at most 200 steps)."""
    from oracle import oracle as O
    from sph_mountain_waves_b200 import cases
    nx, ny, nz = WORKLOADS[sample]
    case = cases.bell_hill_3d(nx, ny, nz, lean=True)
    cores = os.cpu_count() or 1
    O.set_threads(cores)
    o = O.OracleSystem(case.box_min, case.box_max, case.h, case.params)
    o.append(case.fields)
    o.create_cell_list()
    o.step("wcsph", warmup)
    t0 = time.perf_counter()
    done = 0
    while done < steps or (time.perf_counter() - t0 < min_seconds and done < 200):
        o.step("wcsph", 1)
        done += 1
    steps = done
    dt = time.perf_counter() - t0
    n = len(o)
    return {"value": n * steps / dt, "unit": "particle-steps/s", "cores": cores, "kind": "port",
            "sample": f"{sample}: {n} particles x {steps} steps of verlet_step! in {dt:.2f} s, "
                      f"oracle/sph_oracle.c with OpenMP ({cores} threads)",
            "ms_per_step": 1e3 * dt / steps, "n": n, "steps": steps}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference(args.cpu_sample, args.steps, min(args.warmup, 1), min_seconds=0.0)
    line = {
        "impl": "reference", "metric": "particle-steps/s", "value": r["value"], "unit": "particle-steps/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": min(args.warmup, 1), "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic (lattice-initialised)",
        "config": {"workload": args.workload, "cpu_sample": args.cpu_sample, "particles": r["n"],
                   "note": "reference is 100% Julia and julia is not installed: CPU arm = OpenMP C port "
                           "(oracle/sph_oracle.c) of the same verlet_step!, bounded sample of the workload"},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": "particle-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- GPU arm
DUMP_FIELDS = ("h", "x", "m", "v", "rho_p", "rho", "type")   # the carried particle state
DUMP_MAX_PARTICLES = 1 << 19   # x 12 float64 (index + 11 field components) = 48 MiB


def dump_outputs(run, out_dir: str, rank: int, world: int):
    """The particle state the timed steps left, as DIR/<field>.npy in global particle-index order
    (DIR/index.npy holds the indices).  A run larger than DUMP_MAX_PARTICLES is sampled with a
    fixed seed: the same particles for every build, so that two builds compare value for value."""
    import torch.distributed as dist
    n = run.n_global
    if n <= DUMP_MAX_PARTICLES:
        pick = np.arange(n, dtype=np.int64)
    else:
        pick = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_PARTICLES, replace=False))
    want = np.zeros(n, dtype=bool)
    want[pick] = True
    gidx, fields = run.owned_fields(DUMP_FIELDS)
    keep = want[gidx]
    mine = (gidx[keep], {f: a[keep] for f, a in fields.items()})
    parts = [mine]
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, mine)
    if rank != 0:
        return
    idx = np.concatenate([p[0] for p in parts])
    order = np.argsort(idx, kind="stable")
    assert np.array_equal(idx[order], pick), "the ranks do not own each sampled particle exactly once"
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "index.npy", pick.astype(np.float64))
    for f in DUMP_FIELDS:
        np.save(out / f"{f}.npy", np.concatenate([p[1][f] for p in parts])[order].astype(np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist

    from sph_mountain_waves_b200 import cases
    from sph_mountain_waves_b200.slabs import SlabRun

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    is2d = WORKLOADS[args.workload] is None
    nx, ny, nz = (0, 0, 0) if is2d else WORKLOADS[args.workload]
    BYTES = BYTES_2D if is2d else BYTES_3D
    peak_gbs, peak_src = measured_peaks()

    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        if is2d:
            assert world == 1, "the 2D workloads are single-GPU configurations (BASELINE configs 2 and 3)"
            run = SlabRun.whole(getattr(cases, CASES_2D[args.workload])(), device=local, stream=stream.cuda_stream,
                                flags=args.flags)
        else:
            run = SlabRun.bell_hill_3d(nx, ny, nz, rank=rank, world=world, device=local,
                                       stream=stream.cuda_stream, flags=args.flags,
                                       device_gen=args.device_gen)
        if world > 1 and not args.python_transport:
            run.use_library_transport()
        run.create_cell_list()
        n_local = run.n_owned
        n_total = run.n_global

        def barrier():
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
                torch.cuda.synchronize()

        # ---- device-resident throughput ------------------------------------------
        step = (lambda k: run.step(k, overlap=not args.no_overlap)) if world > 1 else run.step
        step(args.warmup)
        # In the timed region only the roofline kernel (pair force + kick) carries event timers: two
        # event records around each of the ~30 launches of a step cost ~0.1 ms of a 6 ms step at
        # N = 8.  The per-kernel breakdown comes from a separate, untimed pass below.
        kname = "wcsph.momentum_fused"
        run.sys.timing(True, prefix=kname)
        run.sys.timing_reset()
        run.sys.count_pairs(True)
        l0 = run.sys.launch_count()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local) as clk:
            ev0.record(stream)
            step(args.steps)
            ev1.record(stream)
            barrier()
        ms = ev0.elapsed_time(ev1)
        launches = run.sys.launch_count() - l0
        rep = run.sys.timing_report()
        if args.dump_outputs:
            dump_outputs(run, args.dump_outputs, rank, world)
        # breakdown pass (not part of any reported throughput)
        nb = max(2, min(args.steps, 5))
        run.sys.timing(True)
        run.sys.timing_reset()
        step(nb)
        barrier()
        rep_all = {k: (v[0] / nb, v[1]) for k, v in run.sys.timing_report().items()}
        run.sys.timing(False)
        # accepted pairs of the force pass (the density pass visits the same set; in slab mode
        # the density pass also covers one ghost column, not counted here)
        pair_list = run.sys.pair_list_info()
        pairs_t = torch.tensor([float(run.sys.pair_count())], dtype=torch.float64, device="cuda")
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(pairs_t, op=dist.ReduceOp.SUM)
        ms_max = float(t.item())
        pairs_force = float(pairs_t.item())
        value = n_total * args.steps / (ms_max * 1e-3)

        # ---- roofline of the dominant kernel (pair force + kick) -----------------
        # (on slabs the overlapped schedule runs it as two launches per step: the edge columns
        # first, "wcsph.momentum_fused_edge", then the interior; one pass = both)
        k_ms, k_calls = rep.get(kname, (0.0, 0))
        k_ms += rep.get(kname + "_edge", (0.0, 0))[0]
        k_calls = max(k_calls, args.steps)
        per_launch_s = (k_ms / max(k_calls, 1)) * 1e-3
        alg_bytes = n_local * BYTES["K_C"]  # the particles this rank owns (ghosts are not its work)
        achieved = alg_bytes / per_launch_s / 1e9 if per_launch_s > 0 else 0.0
        total_kernel_ms = sum(v[0] for v in rep_all.values()) * args.steps
        # DRAM traffic of that kernel per launch: from the committed ncu capture of this very
        # workload/arithmetic on one GPU (never measured under the timed run), else null
        traffic = None
        try:
            tj = json.loads((ROOT / "profiles" / "r02_ncu_traffic.json").read_text())
            rec = tj.get(args.workload, {}).get(f"flags{args.flags}")
            if rec and world == rec["n_gpus"]:
                traffic = (rec["dram_bytes_read"] + rec["dram_bytes_write"]) / 1e9
        except Exception:
            pass
        # the second bound SURVEY.md §8d asks for: the FP64 pipe, against the MEASURED DFMA peak
        # (profiles/microbench/fp64_peak.cu) and with the pipe utilisation ncu saw for this kernel
        fp64 = None
        try:
            pk = json.loads((ROOT / "profiles" / "r02_final_fp64_peak.json").read_text())
            fp64 = {"peak_tflops_measured": pk["fp64_peak_tflops"], "dfma_per_clk_per_sm": pk["dfma_per_clk_per_sm"],
                    "pipe_busy_frac_ncu": 0.447 if not (args.flags & 1) else 0.350,
                    "source": "profiles/r02_final_fp64_peak.json, profiles/r02b_ncu_final_64M_strict.txt "
                              "(sm__inst_executed_pipe_fp64, 64 M particles strict; fast: 9 M particles, "
                              "profiles/r02_ncu_records_8M_fast.txt)"}
        except Exception:
            pass
        roofline = {
            "bound": "hbm", "kernel": kname, "fp64": fp64, "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
            "frac": achieved / peak_gbs, "traffic": traffic, "traffic_unit": "GB per launch (ncu)",
            "alg_gbytes_per_launch": alg_bytes / 1e9, "peak_source": peak_src,
            "alg_bytes_per_particle": BYTES["K_C"], "ms_per_launch": per_launch_s * 1e3,
            "share_of_step": (k_ms / total_kernel_ms) if total_kernel_ms else None,
            "per_kernel_ms_per_step": {k: v[0] for k, v in sorted(rep_all.items())},
            "step_bytes_frac": (n_local * BYTES["step"] * args.steps / (ms * 1e-3) / 1e9) / peak_gbs,
        }

        # ---- the same step with the other arithmetic (fast <-> strict), for reference ----------
        other_ms = None
        if (args.flags & ~1) == 0 and not args.no_strict:
            run.sys.set_flags(args.flags ^ 1)
            step(1)
            barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record(stream)
            step(3)
            s1.record(stream)
            barrier()
            ts = torch.tensor([s0.elapsed_time(s1) / 3], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(ts, op=dist.ReduceOp.MAX)
            other_ms = float(ts.item())
            run.sys.set_flags(args.flags)

        # ---- end to end through the public API with HOST buffers ------------------
        e2e = None
        if not args.no_e2e:
            e2e = run.e2e_cycle(cycles=6, barrier=barrier)   # 6 frame intervals: the copies of one overlap the steps of the next
            te = torch.tensor([e2e["seconds"]], dtype=torch.float64, device="cuda")
            tb = torch.tensor([e2e["h2d_bytes"], e2e["d2h_bytes"]], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
                dist.all_reduce(tb, op=dist.ReduceOp.SUM)
            steps_e2e = e2e["steps"]
            e2e = {"value": n_total * steps_e2e / float(te.item()), "unit": "particle-steps/s",
                   "h2d_bytes_per_step": float(tb[0].item()) / steps_e2e,
                   "d2h_bytes_per_step": float(tb[1].item()) / steps_e2e,
                   "cycle": e2e["what"]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_reference(args.cpu_sample, 3, 1)
        cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        line = {
            "metric": "particle-steps/s", "value": value, "unit": "particle-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic (lattice-initialised, deterministic" +
                    (", generated on the device)" if args.device_gen else ", generated on the host)"),
            "config": {"workload": args.workload, "particles": n_total, "fluid_cells": [nx, ny, nz],
                       "scheme": "wcsph_perturbed_witch verlet_step!" +
                                 (" (2D, wendland2)" if is2d else ", 3D extrusion (wendland3)"),
                       "parallelism": f"x-slabs x{world}",
                       "arithmetic": {0: "strict (no FMA, IEEE div/sqrt; sums bit-identical to the oracle)",
                                      1: "fast (FMA + reciprocals in the closure bodies; exact neighbour set; "
                                         "<=1e-13 rel. of strict per step)",
                                      2: "strict, cell-centric pair-parallel kernel"}.get(args.flags & 3, str(args.flags)),
                       "l2": ("inputs (>= 80 B x particles) far exceed the 126 MB L2; no flush needed"
                              if n_total * 80 > 4 * 126e6 else
                              "SMALL workload: the state (%.0f MB) fits the 126 MB L2, no flush between steps — "
                              "a parity/latency case, not a bandwidth figure" % (n_total * 485 / 1e6)),
                       "pair_interactions_per_s": pairs_force * 2 / (ms_max * 1e-3 / args.steps)
                       if pairs_force else None,
                       "pairs_per_binary_pass": pairs_force,
                       ("fast_arithmetic_ms_per_step" if not (args.flags & 1) else "strict_arithmetic_ms_per_step"): other_ms,
                       "pair_list": pair_list,
                       "halo_exchange": (("overlapped with the interior force pass"
                                          if not (args.flags & 2) and not args.no_overlap else "plain") +
                                         (", ncclSend/ncclRecv inside libsphmw (one group per step)"
                                          if not args.python_transport else ", torch.distributed from Python")
                                         if world > 1 else None),
                       "comm": run.comm_info() if world > 1 and not args.python_transport else None},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
            "clocks": clk.summary(),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

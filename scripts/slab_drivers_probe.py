"""Step time of the hopkins_total and adiabatic flow drivers on one GPU (whole domain) and on N x-slabs.

    torchrun --nproc-per-node N scripts/slab_drivers_probe.py [--n-y 800] [--steps 20] [--warmup 3]

Both drivers run operator by operator (no fused step), on slabs through the library transport
(csrc/slab_comm.cu): hopkins_total with three ghost columns, the adiabatic flow driver ("aflow") with the
open box.  Rank 0 also runs the whole domain on its own GPU (with one rank, only that is measured:
NCCL ranks cannot share a device).  Prints one JSON line: ms/step of both, the host waits per step (cudaStreamSynchronize / cudaEventSynchronize / cudaDeviceSynchronize calls
counted by torch.profiler in a separate short window on rank 0; the timed window runs unprofiled), the
halo exchange counters, and the GPU name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import torch
import torch.distributed as dist

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from sph_mountain_waves_b200 import cases  # noqa: E402
from sph_mountain_waves_b200.slabs import SlabRun  # noqa: E402

MAKE_SYSTEM = ("aflow.find_density", "aflow.find_pressure", "aflow.find_pot_temp", "aflow.find_s",
               "flow.internal_force")   # adiabatic_flow_witch.jl make_system :121-126
WAITS = ("cudaStreamSynchronize", "cudaEventSynchronize", "cudaDeviceSynchronize")


def make_case(driver, n_y):
    if driver == "aflow":
        return cases.aflow_2d(n_y=n_y, dom_length=100e3)
    return cases.hopkins_2d("hopkins_total", n_y=n_y, dom_length=100e3)


def prepare(sys_, driver, create_cell_list):
    create_cell_list()
    if driver == "aflow":
        for op in MAKE_SYSTEM:
            sys_.apply(op)


def timed(step, steps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    step(steps)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / steps


def host_waits(step, steps):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        step(steps)
        torch.cuda.synchronize()
    # the closing synchronize above is the probe's own
    n = sum(1 for e in prof.events() if e.name in WAITS) - 1
    return n / steps


def gpu_info(device):
    q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name(device)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-y", type=float, default=800.0)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--profile-steps", type=int, default=3)
    ap.add_argument("--drivers", default="hopkins_total,aflow")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    result = {"world": world, "n_y": a.n_y, "steps": a.steps, "gpu": gpu_info(local) if rank == 0 else None}
    for driver in a.drivers.split(","):
        case = make_case(driver, a.n_y)
        row = {"particles": case.n}
        # one GPU, whole domain (rank 0)
        if rank == 0:
            s = cases.to_system(case, device=local, capacity=int(case.n * 1.2))
            prepare(s, driver, s.create_cell_list)
            s.step(a.warmup)
            row["whole_ms_per_step"] = timed(s.step, a.steps)
            row["whole_host_waits_per_step"] = host_waits(s.step, a.profile_steps)
            s.close()
        dist.barrier()
        if world < 2:   # NCCL ranks cannot share a device: slabs need one GPU per rank
            result[driver] = row
            continue
        # N slabs through the library transport
        run = SlabRun.from_global_case(case, rank, world, device=local)
        run.use_library_transport(open_box=driver == "aflow")
        prepare(run.sys, driver, run.create_cell_list)
        run.step(a.warmup)
        dist.barrier()
        ms = timed(run.step, a.steps)
        dist.barrier()
        waits = host_waits(run.step, a.profile_steps) if rank == 0 else None
        info = run.comm_info()
        owned = run.n_owned
        gathered = [None] * world
        dist.all_gather_object(gathered, (ms, info, owned))
        row["slabs_ms_per_step"] = max(g[0] for g in gathered)
        row["slabs_ms_per_step_by_rank"] = [round(g[0], 3) for g in gathered]
        row["slabs_host_waits_per_step_rank0"] = waits
        row["exchanges_rank0"] = gathered[0][1]["exchanges"]
        row["renegotiations_rank0"] = gathered[0][1]["renegotiations"]
        row["lost"] = sum(g[1]["lost"] for g in gathered)
        row["owned_by_rank"] = [g[2] for g in gathered]
        result[driver] = row
        run.sys.close()
        dist.barrier()
    if rank == 0:
        line = json.dumps(result)
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as fp:
                fp.write(line + "\n")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

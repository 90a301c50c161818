"""One rank of the adiabatic-flow-on-slabs NCCL test (tests/test_gpu_slabs_more_drivers.py runs it
under torchrun).

The adiabatic flow driver (src/legacy/adiabatic_flow_witch.jl) gains particles at the inflow
(add_new_particles!, :197-208) and loses them through the downstream face of the bounding box
(create_cell_list!'s swap-from-end removal, src/core.jl:72-81); its halo records carry S, P, T and
theta (csrc/halo_record.cuh).  argv: nsteps, driver —
  step       sphmw_step(ctx, "aflow", n) on a context with the library transport and the open box
  operators  the driver's verlet_step! written out with the public calls (apply, aflow_add_new_particles,
             create_cell_list), which are collective on such a context
Rank 0 compares the gathered result, indices included, bit for bit with the whole-domain run on its
own GPU, and checks that particles were both added and removed."""
import os
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from sph_mountain_waves_b200 import cases  # noqa: E402
from sph_mountain_waves_b200.slabs import SlabRun  # noqa: E402

MAKE_SYSTEM = ("aflow.find_density", "aflow.find_pressure", "aflow.find_pot_temp", "aflow.find_s",
               "flow.internal_force")   # make_system :121-126
NAMES = ("x", "v", "Dv", "rho", "m", "P", "theta", "T", "S", "s", "type")


def make_case():
    case = cases.aflow_2d(n_y=20.0, dom_length=30e3, h_m=4e3, a=4e3, U_max=400.0)
    # the conversion line 2.5 dr into the inflow layer: particles convert in the first steps
    case.params["x_inflow"] = -15e3 - 2.5 * case.info["dr"]
    # downstream face 0.3 dr behind the fluid: particles leave within the test
    case.box_max = (15e3 + 0.3 * case.info["dr"], case.box_max[1], 0.0)
    return case


def operator_steps(sys_, create_cell_list, nsteps):
    """verlet_step! of adiabatic_flow_witch.jl:231-243, call by call; returns (added, removed)"""
    added = removed = 0
    for _ in range(nsteps):
        sys_.apply("flow.accelerate")
        sys_.apply("aflow.move")
        added += sys_.aflow_add_new_particles()
        before = len(sys_)
        create_cell_list()
        removed += before - len(sys_)
        sys_.apply("aflow.find_density", True)
        for op in ("aflow.find_s", "aflow.find_pressure", "aflow.entropy_production", "flow.internal_force",
                   "flow.accelerate"):
            sys_.apply(op)
    return added, removed


def same_bits(a, b):
    a, b = np.ascontiguousarray(a, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    nsteps = int(sys.argv[1]) if len(sys.argv) > 1 else 40
    driver = sys.argv[2] if len(sys.argv) > 2 else "step"
    case = make_case()
    failures = []
    run = SlabRun.from_global_case(case, rank, world, device=local)
    run.use_library_transport(open_box=True)
    run.create_cell_list()
    for op in MAKE_SYSTEM:
        run.sys.apply(op)
    added_slabs = 0
    if driver == "step":
        run.step(nsteps)
    else:
        added_slabs, _ = operator_steps(run.sys, run.create_cell_list, nsteps)
    gidx, got = run.owned_fields(NAMES)
    parts = [None] * world
    dist.all_gather_object(parts, (gidx, got, run.comm_info(), added_slabs))
    if rank == 0:
        from util import load_gpu
        whole = load_gpu(case, capacity=2 * case.n)
        n_first = whole.create_cell_list()
        for op in MAKE_SYSTEM:
            whole.apply(op)
        added, removed = operator_steps(whole, whole.create_cell_list, nsteps)
        n_end = len(whole)
        allg = np.concatenate([p[0] for p in parts])
        order = np.argsort(allg, kind="stable")
        lost = [p[2].get("lost") for p in parts]
        print(f"aflow on slabs ({driver}): {case.n} particles, {n_first} after the first cell list, {n_end} after "
              f"{nsteps} steps, {added} added, {removed} removed; lost per rank {lost}", flush=True)
        if not (added > 0 and removed > 0):
            failures.append(f"the run must add and remove particles (added {added}, removed {removed})")
        if driver == "operators" and any(p[3] != added for p in parts):
            failures.append(f"aflow_add_new_particles returned {[p[3] for p in parts]} in total, the whole domain {added}")
        if len(allg) != n_end or not np.array_equal(allg[order], np.arange(n_end)):
            failures.append(f"owned indices are not 0..{n_end - 1} ({len(allg)} particles)")
        else:
            for f in NAMES:
                arr = np.concatenate([p[1][f] for p in parts])[order]
                if not same_bits(arr, whole.field(f)):
                    bad = int(np.sum(np.any(np.atleast_2d(arr.T != whole.field(f).T), axis=0)))
                    failures.append(f"field {f} differs from the whole-domain run in {bad} particles")
        whole.close()
    run.sys.close()
    dist.barrier()
    if rank == 0:
        print("SLAB_AFLOW_OK" if not failures else "SLAB_AFLOW_FAIL " + "; ".join(failures), flush=True)
    dist.destroy_process_group()
    sys.exit(1 if failures else 0)


if __name__ == "__main__":
    main()

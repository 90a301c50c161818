"""The hopkins_total driver (src/current/hopkins_total_witch.jl) and the adiabatic flow driver
(src/legacy/adiabatic_flow_witch.jl) on x-slabs: bitwise equal to the whole-domain run.

hopkins_total keeps three ghost columns (compute_pressure! reads the neighbours' new smoothing
length) and the base halo record with A in row 8.  The adiabatic flow driver's records carry
S, P, T and theta as well (csrc/halo_record.cuh: 17 rows).  Inflow re-seeding numbers the new
particles across ranks, so the adiabatic runs with conversions go through the library transport with
the open box (torchrun, tests/mp/slab_aflow_worker.py); the single-GPU runs here keep the conversion
line out of the box."""
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from sph_mountain_waves_b200 import _capi, cases
from sph_mountain_waves_b200._capi import SphmwError, check
from sph_mountain_waves_b200.slabs import LocalCluster, SlabRun
from util import load_gpu

ROOT = Path(__file__).resolve().parent.parent

MAKE_SYSTEM = ("aflow.find_density", "aflow.find_pressure", "aflow.find_pot_temp", "aflow.find_s",
               "flow.internal_force")   # adiabatic_flow_witch.jl make_system :121-126
AFLOW_FIELDS = ("x", "v", "Dv", "rho", "m", "P", "theta", "T", "S", "s", "type")


def record_width(sys_) -> int:
    w = C.c_int32()
    check(_capi.lib().sphmw_halo_record_width(sys_.ctx, C.byref(w)))
    return w.value


def owners(cluster):
    return [set(r.owned_fields(("m",))[0].tolist()) for r in cluster.runs]


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("U", [20.0, 250.0])
def test_hopkins_total_slabs_bitwise_equal_to_whole_domain(gpu, world, U):
    """hopkins_total_witch.jl:283-308 through step_phase 0/1 around the loop-back transport"""
    case = cases.hopkins_2d("hopkins_total", n_y=16.0, dom_length=120e3, h_m=3000.0, a=10e3, U=U)
    whole = load_gpu(case)
    whole.create_cell_list()
    cluster = LocalCluster([SlabRun.from_global_case(case, r, world) for r in range(world)])
    cluster.create_cell_list()
    assert sum(r.n_owned for r in cluster.runs) == case.n
    own0 = owners(cluster)
    nsteps = 30
    whole.step(nsteps)
    cluster.step(nsteps)
    # walls move and fall in this driver (SURVEY quirk 10): the window must lose nobody, or the
    # comparison below would not be about the same particles
    assert len(whole) == case.n
    assert sum(r.backend.lost for r in cluster.runs) == 0
    names = ("x", "v", "rho", "h", "P", "A", "T", "theta", "m", "type")
    gidx, got = cluster.gather(names)
    assert np.array_equal(gidx, np.arange(case.n))
    for f, a in got.items():
        assert np.array_equal(a, whole.field(f)), f
    if U > 100.0:
        assert owners(cluster) != own0, "no particle changed owner"


def aflow_without_conversions():
    # U_max moves fluid across slab faces within the test; the conversion line lies beyond the box
    case = cases.aflow_2d(n_y=20.0, dom_length=30e3, h_m=4e3, a=4e3, U_max=400.0)
    case.params["x_inflow"] = case.box_max[0] + 10 * case.info["dr"]
    return case


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_aflow_slabs_bitwise_equal_to_whole_domain(gpu, world):
    """adiabatic_flow_witch.jl:231-243 through step_phase 0/1: every field of the 11-field particle of
    the owned particles matches the whole-domain run, with particles changing owner on the way"""
    case = aflow_without_conversions()
    whole = load_gpu(case)
    assert whole.create_cell_list() == case.n
    cluster = LocalCluster([SlabRun.from_global_case(case, r, world) for r in range(world)])
    cluster.create_cell_list()
    assert sum(r.n_owned for r in cluster.runs) == case.n
    for op in MAKE_SYSTEM:
        whole.apply(op)
        for r in cluster.runs:
            r.sys.apply(op)
    own0 = owners(cluster)
    nsteps = 40
    whole.step(nsteps)
    cluster.step(nsteps)
    assert len(whole) == case.n
    assert sum(r.backend.lost for r in cluster.runs) == 0
    assert owners(cluster) != own0, "no particle changed owner"
    gidx, got = cluster.gather(AFLOW_FIELDS)
    assert np.array_equal(gidx, np.arange(case.n))
    for f, a in got.items():
        assert np.array_equal(a, whole.field(f)), f


@pytest.mark.gpu
def test_aflow_step_phase_refuses_a_converting_particle(gpu):
    """the successors' global indices need the converting particles of all ranks: the host-driven
    step fails loudly instead of skipping them"""
    case = cases.aflow_2d(n_y=20.0, dom_length=30e3, h_m=4e3, a=4e3, U_max=40.0)
    case.params["x_inflow"] = -15e3 - 2.5 * case.info["dr"]   # the inflow layer converts at once
    cluster = LocalCluster([SlabRun.from_global_case(case, r, 2) for r in range(2)])
    cluster.create_cell_list()
    with pytest.raises(SphmwError, match="open box"):
        cluster.runs[0].backend.pre()


@pytest.mark.gpu
def test_hopkins_total_on_a_two_column_slab_is_refused(gpu):
    case = cases.hopkins_2d("hopkins_total", n_y=16.0, dom_length=120e3)
    case.scheme = "wcsph"          # sliced like a WCSPH case: two ghost columns
    run = SlabRun.from_global_case(case, 0, 2)
    run.sys.T.scheme = "hopkins_total"
    with pytest.raises(SphmwError, match="three ghost columns"):
        run.backend.pre()
        run.backend.post()


@pytest.mark.gpu
def test_aflow_add_new_particles_needs_the_library_transport(gpu):
    case = aflow_without_conversions()
    run = SlabRun.from_global_case(case, 0, 2)
    with pytest.raises(SphmwError, match="library transport"):
        run.sys.aflow_add_new_particles()
    with pytest.raises(SphmwError, match="library transport"):
        run.sys.flow_add_new_particles()


@pytest.mark.gpu
def test_halo_record_width_per_context(gpu):
    """13 doubles (the base record) unless the context holds the entropy S: 17"""
    wide = dict(n_y=16.0, dom_length=120e3)
    for case, want in ((cases.mountain_wave_2d(**wide), 13), (cases.hopkins_2d("hopkins_total", **wide), 13),
                       (cases.flow_2d(n_y=20.0, dom_length=30e3, h_m=4e3, a=4e3), 13), (aflow_without_conversions(), 17)):
        s = load_gpu(case)
        s._flush()   # the fields reach the device, then the width is fixed by its first use
        assert record_width(s) == want, case.name
        s.close()
        run = SlabRun.from_global_case(case, 0, 2)
        assert run.backend.width == record_width(run.sys) == want, case.name
        run.sys.close()


def aflow_with_inflow_and_outflow():
    # the conversion line 2.5 dr into the inflow layer, the downstream face 0.3 dr behind the fluid:
    # particles are added and removed within the test
    case = cases.aflow_2d(n_y=20.0, dom_length=30e3, h_m=4e3, a=4e3, U_max=400.0)
    case.params["x_inflow"] = -15e3 - 2.5 * case.info["dr"]
    case.box_max = (15e3 + 0.3 * case.info["dr"], case.box_max[1], 0.0)
    return case


def aflow_operator_steps(sys_, nsteps):
    """verlet_step! of adiabatic_flow_witch.jl:231-243, call by call; returns (added, removed)"""
    added = removed = 0
    for _ in range(nsteps):
        sys_.apply("flow.accelerate")
        sys_.apply("aflow.move")
        added += sys_.aflow_add_new_particles()
        before = len(sys_)
        sys_.create_cell_list()
        removed += before - len(sys_)
        sys_.apply("aflow.find_density", True)
        for op in ("aflow.find_s", "aflow.find_pressure", "aflow.entropy_production", "flow.internal_force",
                   "flow.accelerate"):
            sys_.apply(op)
    return added, removed


@pytest.mark.gpu
def test_aflow_communicator_created_before_the_upload(gpu):
    """the Julia shim's order: sphmw_create, sphmw_comm_init (+ open box), and only then the particles.
    The record width follows from the uploaded fields at the first exchange, so the adiabatic driver's
    literal verlet_step! runs — here on a one-rank communicator over the whole column range, with
    inflow and outflow, bitwise equal to the whole-domain run, indices included"""
    import torch  # noqa: F401  (loads the NCCL library the transport opens)
    from sph_mountain_waves_b200.slabs import LibSlabBackend, plan_slab
    case = aflow_with_inflow_and_outflow()
    plan = plan_slab(case.box_min, case.box_max, case.h, 0, 1)
    slab = cases.to_system(case, slab=(plan.lo, plan.hi), capacity=2 * case.n)   # fields staged on the host
    lib = _capi.lib()
    ident = (C.c_ubyte * 128)()
    check(lib.sphmw_comm_unique_id(ident))
    check(lib.sphmw_comm_init(slab.ctx, 0, 1, bytes(ident), 4096))
    check(lib.sphmw_comm_open_box(slab.ctx, 1))
    slab._flush()                                                             # the upload
    check(lib.sphmw_set_index(slab.ctx, _capi.ptr(np.arange(case.n, dtype=np.int64)), case.n))
    whole = load_gpu(case, capacity=2 * case.n)
    n_first = whole.create_cell_list()
    slab.create_cell_list()
    assert record_width(slab) == 17
    for op in MAKE_SYSTEM:
        whole.apply(op)
        slab.apply(op)
    nsteps = 40
    added, removed = aflow_operator_steps(whole, nsteps)
    added_slab, _ = aflow_operator_steps(slab, nsteps)
    assert added > 0 and removed > 0, (added, removed)
    assert added_slab == added
    n_end = n_first + added - removed
    assert len(whole) == n_end
    gidx, got = SlabRun(slab, plan, case.n, LibSlabBackend(slab, plan, 4096)).owned_fields(AFLOW_FIELDS)
    order = np.argsort(gidx, kind="stable")
    assert np.array_equal(gidx[order], np.arange(n_end))
    for f, a in got.items():
        assert np.array_equal(a[order], whole.field(f)), f


def _gpus():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


def _torchrun(world, port, script, *args):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), str(ROOT / "tests" / "mp" / script), *args]
    return subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=str(ROOT))


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("driver", ["step", "operators"])
def test_aflow_on_slabs_with_inflow_and_outflow(world, driver):
    """the adiabatic flow driver through the library transport with the open box: inflow re-seeding
    (new global indices in the reference's order) and outflow by removal, across ranks, bitwise equal
    to the whole-domain run — through sphmw_step(ctx, "aflow", n) and through the public
    operator-by-operator calls (tests/mp/slab_aflow_worker.py)"""
    if _gpus() < world:
        pytest.skip(f"needs {world} GPUs")
    r = _torchrun(world, 33500 + (os.getpid() % 2000), "slab_aflow_worker.py", "40", driver)
    assert r.returncode == 0 and "SLAB_AFLOW_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.gpu
def test_hopkins_total_through_the_nccl_transports():
    """sphmw_step(ctx, "hopkins_total", n) on contexts with a communicator, and step_phase 0/1 around
    torch.distributed, bitwise equal to the whole-domain run (tests/mp/slab_nccl_worker.py)"""
    if _gpus() < 2:
        pytest.skip("needs 2 GPUs")
    r = _torchrun(2, 34500 + (os.getpid() % 2000), "slab_nccl_worker.py", "12", "0", "hopkins_total")
    assert r.returncode == 0 and "SLAB_NCCL_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]

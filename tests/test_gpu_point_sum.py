"""Point sums on the device (sphmw_point_sum, ParticleSystem.point_sum / interpolate): the sum(sys, f, x)
of src/core.jl:240-291 at points that are not particles.  Strict arithmetic: every op equals the CPU
restatement (tests/c/point_sum_oracle.c) with ==, after a cell-list build, after fused steps and in the x-chunked cell order; the
call changes no state."""
import numpy as np
import pytest

import point_cases as pc
import point_oracle
from sph_mountain_waves_b200 import _capi
from sph_mountain_waves_b200._capi import SphmwError
from util import load_gpu, n_mismatch

pytestmark = pytest.mark.gpu

TILES = 64
STATE = ["x", "v", "m", "rho", "rho_p", "h", "type", "P", "theta", "T", "Dv"]


def restated(case, s, pts, ops, extra=()):
    """the CPU restatement on the device's downloaded state, building its own cell list"""
    fields = {f: s.field(f) for f in ("x", "v", "m", "rho", "rho_p") + tuple(extra)}
    return point_oracle.point_sum(case.box_min, case.box_max, case.h, fields, pts, ops)


def assert_equals_restatement(case, s, pts):
    ops = pc.ops_for(case)
    got = s.point_sum(pts, ops)
    want = restated(case, s, pts, ops)
    for k, op in enumerate(ops):
        assert n_mismatch(got[k], want[k]) == 0, op
    assert np.isnan(got[0]).sum() >= 4 and (got[0] > 0).sum() > len(pts) // 2
    return got


CASES = {"witch2d": pc.witch_2d, "hill3d": pc.hill_3d, "hex2d": pc.hex_2d}


@pytest.mark.parametrize("name", list(CASES))
def test_point_sum_equals_the_restatement_after_build_steps_and_in_both_cell_orders(gpu, name):
    case = CASES[name]()
    pts = pc.sample_points(case)
    s = load_gpu(case)
    s.create_cell_list()
    assert_equals_restatement(case, s, pts)
    s.step(5)
    assert_equals_restatement(case, s, pts)
    s.set_flags(TILES)  # the x-chunked physical cell order
    assert_equals_restatement(case, s, pts)
    s.close()


@pytest.mark.parametrize("name", ["hill3d", "witch2d"])
def test_a_million_random_points_come_back_in_caller_order(gpu, name):
    """2^20 points in random order exercise the sort by home cell; results are in the caller's order"""
    case = CASES[name]()
    rng = np.random.default_rng(11)
    lo, hi = np.array(case.box_min), np.array(case.box_max)
    pts = lo + rng.random((1 << 20, 3)) * (hi - lo)
    if case.dim == 2:
        pts[:, 2] = 0.0
    pts[::97] = np.nan
    s = load_gpu(case)
    s.create_cell_list()
    s.step(2)
    assert_equals_restatement(case, s, pts)
    s.close()


def test_cuda_tensors_in_and_out_equal_host_buffers(gpu):
    import torch
    case = pc.hill_3d()
    pts = pc.sample_points(case)
    s = load_gpu(case)
    s.create_cell_list()
    s.step(1)
    ops = pc.ops_for(case)
    host = s.point_sum(pts, ops)
    dev = s.point_sum(torch.from_numpy(pts).cuda(), ops)
    assert dev.is_cuda and tuple(dev.shape) == host.shape
    assert n_mismatch(dev.cpu().numpy(), host) == 0
    ih = s.interpolate(pts, ["v[0]", "rho_p"])
    idev = s.interpolate(torch.from_numpy(pts).cuda(), ["v[0]", "rho_p"])
    for f in ih:
        assert n_mismatch(idev[f].cpu().numpy(), ih[f]) == 0
        with np.errstate(invalid="ignore", divide="ignore"):
            assert n_mismatch(ih[f], np.where(host[2] == 0, np.nan, host[4 if f == "v[0]" else 6] / host[2])) == 0
    assert np.isnan(ih["v[0]"]).any() and np.isfinite(ih["v[0]"]).sum() > len(pts) // 2
    s.close()


def test_stale_theta_is_brought_up_to_date(gpu):
    """after a fused step theta is stale; the call rebuilds it first (as sphmw_reduce does)"""
    case = pc.witch_2d()
    pts = pc.sample_points(case)
    s = load_gpu(case)
    s.create_cell_list()
    s.step(2)
    before = s.point_sum(pts, ["VW*theta", "VW*θ"])
    theta = s.field("theta")                     # explicit materialisation
    after = s.point_sum(pts, ["VW*theta"])
    assert n_mismatch(before[0], after[0]) == 0 and n_mismatch(before[1], after[0]) == 0
    assert n_mismatch(theta, s.field("theta")) == 0
    assert n_mismatch(after, restated(case, s, pts, ["VW*theta"], extra=("theta",))) == 0
    assert np.nanmax(np.abs(after)) > 0
    s.close()


@pytest.mark.parametrize("name", ["witch2d", "hill3d"])
def test_no_side_effects(gpu, name):
    """a point sum changes no field, and the following steps equal a control run's bit for bit with the
    same number of launches"""
    case = CASES[name]()
    pts = pc.sample_points(case)
    runs = []
    for probe in (False, True):
        s = load_gpu(case)
        s.create_cell_list()
        s.step(2)
        before = {f: s.field(f) for f in STATE}
        if probe:
            s.point_sum(pts, pc.ops_for(case))
            s.point_sum(pts, ["VW*theta", "mW*T", "VW*Dv[1]"])
            for f in STATE:
                assert n_mismatch(s.field(f), before[f]) == 0, f
        l0 = s.launch_count()
        s.step(3)
        runs.append(({f: s.field(f) for f in STATE}, s.launch_count() - l0))
        s.close()
    assert runs[0][1] == runs[1][1]
    for f in STATE:
        assert n_mismatch(runs[0][0][f], runs[1][0][f]) == 0, f


def test_refusals(gpu):
    case = pc.witch_2d()
    pts = pc.sample_points(case)[:16]
    s = load_gpu(case)
    with pytest.raises(SphmwError) as e:                  # no cell list yet
        s.point_sum(pts, ["count"])
    assert e.value.code == _capi.E_STATE
    s.create_cell_list()
    assert s.point_sum(np.zeros((0, 3)), ["count"]).shape == (1, 0)
    for ops, code in ((["count", "W"], _capi.E_UNSUPPORTED_OP), (["mWx"], _capi.E_UNSUPPORTED_OP),
                      (["VW*nope"], _capi.E_UNKNOWN_FIELD), ([], _capi.E_INVALID), (["count"] * 9, _capi.E_INVALID),
                      (["VW*v[2]"], _capi.E_INVALID), (["VW*v"], _capi.E_INVALID)):
        with pytest.raises(SphmwError) as e:
            s.point_sum(pts, ops)
        assert e.value.code == code, ops
    assert s.point_sum(pts, ["count"] * 8).shape == (8, 16)
    s.apply("wcsph.move")
    with pytest.raises(SphmwError) as e:
        s.point_sum(pts, ["count"])
    assert e.value.code == _capi.E_STATE
    s.close()

    from sph_mountain_waves_b200 import cases
    from sph_mountain_waves_b200.slabs import plan_slab
    plan = plan_slab(case.box_min, case.box_max, case.h, 0, 2)
    slab = cases.to_system(case, slab=(plan.lo, plan.hi), capacity=2 * case.n)
    with pytest.raises(SphmwError) as e:
        slab.point_sum(pts, ["count"])
    assert e.value.code == _capi.E_STATE and "slab" in str(e.value)
    slab.close()

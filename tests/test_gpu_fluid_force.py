"""The force pass of the fused WCSPH step evaluates the pair sums of fluid particles only
(csrc/pair_list.cuh k_binary_list_fluid, over the fluid work list of each cell-list build): walls and the
mountain keep their velocity whatever their neighbours do, so skipping their pairs must not change a bit
of any field, nor the pair count."""
import numpy as np
import pytest

from sph_mountain_waves_b200 import cases
from util import bits_equal, field_err, load_gpu, load_oracle

pytestmark = pytest.mark.gpu

FAST_MATH, NO_LIST = 1, 4
FIELDS = ["x", "v", "h", "rho", "rho_p", "P", "type"]


def small_2d():
    return cases.mountain_wave_2d(n_y=24.0, dom_length=80e3, h_m=3000.0, a=10e3, U=20.0)


def small_3d():
    return cases.bell_hill_3d(24, 12, 10, h_m=3000.0, a=8e3, U=20.0)


def run(case, flags, calls, edit=None):
    s = load_gpu(case, flags=flags)
    s.create_cell_list()
    s.count_pairs(True)
    for k, n in enumerate(calls):
        if edit and k == 1:
            edit(s)
        s.step(n)
    out = ({f: s.field(f) for f in FIELDS}, s.pair_count())
    s.close()
    return out


@pytest.mark.parametrize("make", [small_2d, small_3d])
@pytest.mark.parametrize("arith", [0, FAST_MATH])
def test_one_call_equals_one_step_calls_and_the_oracle(gpu, make, arith):
    """one call of six steps == six calls of one step == the cell walk (every particle's pairs) bit for
    bit; the pair count of the last force pass is the oracle's"""
    case = make()
    fluid = case.fields["type"] == case.params["fluid"]
    assert 0 < fluid.sum() < case.n
    walk = run(case, NO_LIST | arith, [6])
    one = run(case, arith, [6])
    single = run(case, arith, [1] * 6)
    o = load_oracle(case)
    o.create_cell_list()
    o.step("wcsph", 6)
    for got in (one, single):
        assert got[1] == walk[1] == o.pair_count() > 0
        for f in FIELDS:
            assert bits_equal(got[0][f], walk[0][f]), f
    for f in ("x", "v", "rho", "h"):
        assert field_err(case, f, one[0][f], o.field(f), nsteps=6) <= 1e-10, f


@pytest.mark.parametrize("make", [small_2d, small_3d])
def test_type_change_between_calls(gpu, make):
    """set_field("type") between two calls: the next cell-list build makes a new fluid work list, so the
    force pass follows the new types exactly as the cell walk does"""
    case = make()

    def edit(s):
        t = s.field("type")
        fluid = np.flatnonzero(t == case.params["fluid"])
        other = t[t != case.params["fluid"]][0]
        t[fluid[::5]] = other
        s.set_field("type", t)

    walk = run(case, NO_LIST, [3, 3], edit)
    one = run(case, 0, [3, 3], edit)
    assert one[1] == walk[1] > 0
    for f in FIELDS:
        assert bits_equal(one[0][f], walk[0][f]), f
    assert np.sum(one[0]["type"] == case.params["fluid"]) < np.sum(case.fields["type"] == case.params["fluid"])


def test_particle_leaving_the_box_mid_call(gpu):
    """a fluid particle that leaves the box during a multi-step call is removed as before: the cell
    list and the fluid work list shrink with it, and the result equals the cell walk and the oracle"""
    case = small_3d()
    fields = {k: np.array(v, copy=True) for k, v in case.fields.items()}
    fluid = np.flatnonzero(fields["type"] == case.params["fluid"])
    p = fluid[len(fluid) // 2]
    # leaves through the top face within a few steps
    fields["v"][p, 1] = (case.box_max[1] - fields["x"][p, 1]) / (2.5 * case.params["dt"])
    case = cases.Case(case.name, case.scheme, case.dim, case.box_min, case.box_max, case.h, case.params, fields,
                      case.info)
    walk = run(case, NO_LIST, [5])
    one = run(case, 0, [5])
    assert len(one[0]["x"]) == len(walk[0]["x"]) == case.n - 1
    assert one[1] == walk[1]
    for f in FIELDS:
        assert bits_equal(one[0][f], walk[0][f]), f
    o = load_oracle(case)
    o.create_cell_list()
    o.step("wcsph", 5)
    assert len(o) == case.n - 1
    for f in ("x", "v", "rho"):
        assert field_err(case, f, one[0][f], o.field(f), nsteps=5) <= 1e-10, f


# ---- cell keys from the advance: in a whole-domain call of n steps, the force pass of steps 1..n-1 also
# writes the next cell list's key of each drifted particle, and the next build skips k_keys ----------------

def test_cell_keys_after_a_call_equal_a_fresh_build(gpu, monkeypatch):
    """the cell list a multi-step call leaves behind was sorted by keys from the advance: they equal a
    fresh build's and those of a call whose every build runs k_keys.  (Not compared with the oracle: the
    strict positions agree with it to 1e-10 only, and a lattice particle that sits on a cell face can
    land on either side of it.)"""
    case = small_3d()
    s = load_gpu(case)
    s.create_cell_list()
    s.timing(True)
    s.step(5)
    keys_launches = s.timing_report()["cell_keys"][1]
    keys = s.cell_keys()
    s.create_cell_list()
    fresh = s.cell_keys()
    s.close()
    monkeypatch.setenv("SPHMW_NO_FUSED_ADVANCE", "1")
    p = load_gpu(case)
    p.create_cell_list()
    p.step(5)
    plain = p.cell_keys()
    p.close()
    assert np.array_equal(keys, fresh)
    assert np.array_equal(keys, plain)
    assert keys_launches == 1  # the first build of the call; the other four took the advance's keys


def test_set_field_x_between_calls_is_rekeyed(gpu, monkeypatch):
    """positions set between two calls are keyed afresh: the result equals a run without the folded
    advance (every build runs k_keys)"""
    case = small_3d()

    def edit(s):
        x = s.field("x")
        x[::7, 0] += 0.6 * case.h
        s.set_field("x", x)

    one = run(case, 0, [3, 3], edit)
    monkeypatch.setenv("SPHMW_NO_FUSED_ADVANCE", "1")
    plain = run(case, 0, [3, 3], edit)
    assert one[1] == plain[1] > 0
    for f in FIELDS:
        assert bits_equal(one[0][f], plain[0][f]), f

"""sphmw_reduce against exact values: math.fsum for sums, exact max, an extended-precision |v|.

The reduction is a fixed tree: 1024 blocks of 256 threads, each thread adding its grid-stride
values in order (ceil(n / 262144) additions), then 5 shuffle levels in the warp and 3 over the 8
warps of the block; a second launch of one block of 1024 threads adds the 1024 block results
with 5 + 5 levels.  Every value therefore passes through at most
    d = ceil(n / 262144) + 18
additions, and the FP64 sum s of values x_i satisfies |s - sum x_i| <= gamma_d * sum |x_i|,
gamma_d = d u / (1 - d u), u = 2^-53 (Higham, Accuracy and Stability, eq. 4.3)."""
import math

import numpy as np
import pytest

from sph_mountain_waves_b200 import cases
from sph_mountain_waves_b200._capi import E_STATE, E_UNKNOWN_FIELD, SphmwError
from sph_mountain_waves_b200.slabs import LocalCluster, SlabRun
from util import load_gpu

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
SIZES = [1, 31, 32, 33, 255, 256, 257, 262143, 262144, 262145, 2 ** 20 + 3]
CAPACITY = 2 ** 20 + 8


def gamma(n):
    d = -(-n // 262144) + 18
    return d * U / (1 - d * U)


@pytest.fixture(scope="module")
def sys2d(gpu):
    s = load_gpu(cases.mountain_wave_2d(n_y=12.0, dom_length=30e3), capacity=CAPACITY)
    s._flush()
    yield s
    s.close()


@pytest.fixture(scope="module")
def sys3d(gpu):
    s = load_gpu(cases.bell_hill_3d(10, 8, 6, h_m=3000.0, a=4e3, U=25.0), capacity=CAPACITY)
    s._flush()
    yield s
    s.close()


def with_values(s, name, a):
    s.resize(0)                # a context only shrinks to 0
    s.resize(len(a))
    s.set_field(name, a)
    return s


def wide_values(n, seed):
    """magnitudes from 1e-300 to 1e300, random signs, and runs of values that cancel exactly"""
    rng = np.random.default_rng(seed)
    a = rng.choice([-1.0, 1.0], n) * 10.0 ** rng.uniform(-300, 300, n)
    if n >= 8:
        k = n // 4
        a[k:2 * k:2] = -a[k + 1:2 * k + 1:2][: len(a[k:2 * k:2])]
    return a


@pytest.mark.parametrize("n", SIZES)
def test_sum_within_the_tree_bound(sys2d, n):
    for seed, a in enumerate([wide_values(n, n), np.random.default_rng(n).normal(size=n)]):
        s = with_values(sys2d, "rho", a)
        got = s.reduce("sum:rho")
        exact = math.fsum(a)
        bound = gamma(n) * math.fsum(np.abs(a))
        assert abs(got - exact) <= bound, (n, seed, got, exact, bound)


@pytest.mark.parametrize("n", SIZES)
def test_max_is_exact(sys2d, n):
    a = wide_values(n, 7 * n)
    assert with_values(sys2d, "rho", a).reduce("max:rho") == a.max()
    neg = -np.abs(a) - 1.0
    assert with_values(sys2d, "rho", neg).reduce("max:rho") == neg.max()


@pytest.mark.parametrize("n,where", [(257, 0), (257, 256), (33, 32), (2 ** 20 + 3, 262144 + 5), (2 ** 20 + 3, 2 ** 20 + 2)],
                         ids=["first", "last", "partial-warp", "second-stride-round", "last-large"])
def test_max_propagates_nan(sys2d, n, where):
    a = np.random.default_rng(where).normal(size=n)
    a[where] = np.nan
    assert math.isnan(with_values(sys2d, "rho", a).reduce("max:rho"))


def test_max_infinities(sys2d):
    a = np.random.default_rng(3).normal(size=1000)
    a[500] = np.inf
    assert with_values(sys2d, "rho", a).reduce("max:rho") == math.inf
    assert with_values(sys2d, "rho", np.full(1000, -np.inf)).reduce("max:rho") == -math.inf


@pytest.mark.parametrize("n", [1, 2, 33, 257, 262145, 2 ** 20 + 3])
def test_max_of_signed_zeros_is_positive_zero(sys2d, n):
    """Julia's max orders -0.0 below +0.0; any mix of zeros gives +0.0 wherever they sit"""
    rng = np.random.default_rng(n)
    for a in (rng.choice([-0.0, 0.0], n), np.r_[np.full(n - 1, -0.0), 0.0] if n > 1 else np.array([0.0]),
              np.r_[0.0, np.full(n - 1, -0.0)], -np.abs(rng.normal(size=n)) * 0.0):
        got = with_values(sys2d, "rho", a).reduce("max:rho")
        want = 0.0 if (np.signbit(a) == False).any() else -0.0   # noqa: E712
        assert got == 0.0 and math.copysign(1.0, got) == math.copysign(1.0, want), (n, got)


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("n", [1, 257, 262145])
def test_speeds(sys2d, sys3d, dim, n):
    s = sys2d if dim == 2 else sys3d
    rng = np.random.default_rng(n + dim)
    v = rng.normal(scale=20.0, size=(n, 3))
    if dim == 2:
        v[:, 2] = 0.0
    with_values(s, "v", v)
    speed64 = np.sqrt(v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1] + v[:, 2] * v[:, 2])   # algebra.jl:49-60
    assert s.reduce("max_speed") == speed64.max()
    vl = v.astype(np.longdouble)
    speed = np.sqrt((vl * vl).sum(1))
    mean = speed.sum() / n
    # per value: the FP64 |v| is within 3 u (2 or 3 roundings in the sum of squares, 1 in sqrt)
    bound = (gamma(n) + 3 * U) * float(speed.sum()) / n + U * float(mean)
    assert abs(np.longdouble(s.reduce("avg_speed")) - mean) <= bound


def test_sum_of_stale_theta_after_a_fused_step(gpu):
    """theta is stale after sphmw_step; reduce rebuilds it first"""
    case = cases.mountain_wave_2d(n_y=24.0, dom_length=80e3, h_m=3000.0, a=10e3, U=20.0)
    s = load_gpu(case)
    s.create_cell_list()
    s.step(2)
    got = s.reduce("sum:theta")
    th = s.field("theta")
    assert abs(got - math.fsum(th)) <= gamma(len(th)) * math.fsum(np.abs(th))
    assert got != math.fsum(case.fields["theta"])
    s.close()


def test_unwritten_vector_and_empty(sys2d):
    s = with_values(sys2d, "rho", np.ones(100))
    assert s.reduce("sum:S") == 0.0 and s.reduce("max:S") == 0.0      # never written: constructor zero
    assert s.reduce("count") == 100.0
    for what in ("sum:v", "max:x"):
        with pytest.raises(SphmwError) as e:
            s.reduce(what)
        assert e.value.code == E_UNKNOWN_FIELD
    s.resize(0)
    for what in ("count", "sum:rho", "max:rho", "avg_speed", "max_speed"):
        assert s.reduce(what) == 0.0


def test_slab_contexts_are_refused(gpu):
    case = cases.bell_hill_3d(24, 12, 10, h_m=3000.0, a=8e3, U=20.0)
    cluster = LocalCluster([SlabRun.from_global_case(case, r, 2) for r in range(2)])
    try:
        cluster.create_cell_list()
        for run in cluster.runs:
            for what in ("count", "sum:rho", "max:rho", "avg_speed", "max_speed"):
                with pytest.raises(SphmwError) as e:
                    run.sys.reduce(what)
                assert e.value.code == E_STATE and "sphmw_slab_counts" in str(e.value)
    finally:
        for run in cluster.runs:
            run.sys.close()

"""GPU: the bracket of the centralized optimum (revs_central_bracket) against the numpy model of tests/central_ref.py, on
mixed zones, on reference-shaped feeders at the bench's limits and on a tree-only zone; the kept schedule's network
check, pipelines, determinism, independence from the ADMM run and argument errors."""
import ctypes

import numpy as np
import pytest

import central_ref as CR
import network_ref as NR
import repair_ref as RR
from revs_admm_b200.feeder import population, radial_feeder, synthetic_homes, synthetic_tariff
from test_gpu_network import BENCH, _mixed_zones, _solved, _solver

pytestmark = pytest.mark.gpu

LIMITS = dict(vset=BENCH["vset"], vhigh=BENCH["vhigh"])


def _vhigh(zones, hm, factor):
    """vhigh (vset = 1) whose limit is `factor` times the largest drop of the base load alone."""
    return float(np.sqrt(1.0 + factor * NR.network_check(zones, hm["load"])["drop"].max()))


def _ready(lib, zones, hm, cost, T, cls=None):
    s = _solver(lib, zones, T, cls=cls)
    s.set_homes(**hm)
    s.set_tariff(cost)
    return s


def _check_equal(got, ref, T):
    assert np.array_equal(got["zone_info"], ref["zone_info"])
    assert np.array_equal(got["zone_bounds"], ref["zone_bounds"])
    assert np.array_equal(RR.unpack(got["mask"], T), ref["bits"])
    assert np.array_equal(got["P_sch"], ref["P_sch"])


@pytest.mark.parametrize("T", [24, 37, 96])
def test_matches_model_on_mixed_zones(gpu_lib, T):
    zones = _mixed_zones(T)
    hm = synthetic_homes(sum(z.n_res for z in zones), T, seed=T)
    cost = synthetic_tariff(T)
    kw = dict(vset=1.0, vhigh=_vhigh(zones, hm, 1.3), iters=40)
    with _ready(gpu_lib, zones, hm, cost, T) as s:
        got = s.central_bracket(mask=True, **kw)
    _check_equal(got, CR.bracket(zones, hm, cost, **kw), T)
    assert sum(got["zones_status"][1:]) > 0 and got["zone_info"][:, 1].sum() > 0


def _refshape(n):
    trees, hm, cost, sizes, T = population("refshape", n, seed=0)
    return trees, hm, cost, T


def test_reference_shaped_feeders(gpu_lib):
    import bench
    trees, hm, cost, T = _refshape(3)
    with _ready(gpu_lib, trees, hm, cost, T) as s:
        got = s.central_bracket(mask=True, iters=30, **LIMITS)
        chk = s.network_check("central", zones=True, **LIMITS)
    _check_equal(got, CR.bracket(trees, hm, cost, iters=30, **LIMITS), T)
    st = got["zone_info"][:, 0]
    assert (st == 1).any()
    assert (chk["zone_worst"][st <= 1, 1] <= 1e-9).all()
    _, lb0, _ = bench.objective_check(trees, hm, cost, got["P_sch"], T)
    assert got["lb"] >= lb0 * (1 - 1e-12)


def test_tree_only_zone_uses_the_global_state(gpu_lib):
    T = 96
    zones = [radial_feeder(2300, seed=3, r_scale=0.07)]
    hm = synthetic_homes(2300, T, seed=4)
    cost = synthetic_tariff(T)
    kw = dict(vset=1.0, vhigh=_vhigh(zones, hm, 1.3), iters=10)
    with _ready(gpu_lib, zones, hm, cost, T) as s:
        got = s.central_bracket(mask=True, **kw)
    _check_equal(got, CR.bracket(zones, hm, cost, **kw), T)
    assert got["zone_info"][0, 0] > 0


def test_pipelines_equal_one_solver(gpu_lib):
    trees, hm, cost, T = _refshape(6)
    kw = dict(mask=True, iters=20, **LIMITS)
    with _ready(gpu_lib, trees, hm, cost, T) as a:
        ra = a.central_bracket(**kw)
        na = a.network_check("central", zones=True, **LIMITS)
    with _ready(gpu_lib, trees, hm, cost, T, cls=lambda sizes, T: gpu_lib.PipelinedSolver(sizes, T, pipelines=4)) as b:
        assert len(b.parts) == 4
        rb = b.central_bracket(**kw)
        nb = b.network_check("central", zones=True, **LIMITS)
    for k in ("P_sch", "mask", "zone_bounds", "zone_info"):
        assert np.array_equal(ra[k], rb[k]), k
    for k in ("lb", "lb_bracketed", "ub", "gap", "zones_status"):
        assert ra[k] == rb[k], k
    assert na["summary"] == nb["summary"] and np.array_equal(na["zone_worst"], nb["zone_worst"])


def test_deterministic_and_independent_of_the_admm_run(gpu_lib):
    trees, hm, cost, T = _refshape(2)
    kw = dict(mask=True, iters=20, **LIMITS)
    with _ready(gpu_lib, trees, hm, cost, T) as s:
        n0 = s.stats()["kernel_launches"]
        a = s.central_bracket(**kw)                                # before any ADMM run
        assert s.stats()["kernel_launches"] > n0
        s.solve_admm(**BENCH)
        before, est = s.results(), s.estimate()
        rep = s.repair_schedule(mask=True, **LIMITS)
        b = s.central_bracket(**kw)
        for k in ("P_sch", "mask", "zone_bounds", "zone_info"):
            assert a[k].tobytes() == b[k].tobytes(), k
        after, est2 = s.results(), s.estimate()
        for k in before:
            assert np.array_equal(before[k], after[k]), k
        assert all(np.array_equal(x, y) for x, y in zip(est, est2))
        rep2 = s.repair_schedule(mask=True, **LIMITS)
        for k in ("P_sch", "mask", "zone_info"):
            assert np.array_equal(rep[k], rep2[k]), k
        chk = s.network_check("repaired", zones=True, **LIMITS)
        s.central_bracket(**kw)
        assert np.array_equal(chk["zone_worst"], s.network_check("repaired", zones=True, **LIMITS)["zone_worst"])


def test_argument_errors(gpu_lib):
    T = 24
    zones = _mixed_zones(1)[:2]
    hm = synthetic_homes(sum(z.n_res for z in zones), T, seed=2)
    cost = synthetic_tariff(T)

    def code(fn, c=1):
        with pytest.raises(gpu_lib.RevsError) as e:
            fn()
        assert e.value.code == c, str(e.value)
        return str(e.value)

    lib = gpu_lib._cabi.load()
    assert lib.revs_central_bracket(None, 1.0, 1.05, 1e-9, 10, None, None, 1, None, None) == 1
    with gpu_lib.Solver([z.n_res for z in zones], T) as s:
        s.set_feeder_tree(0, zones[0].parent, zones[0].r, zones[0].res_node)
        s.set_sensitivity(1, np.eye(zones[1].n_res) * 1e-3)
        s.set_homes(**hm)
        s.set_tariff(cost)
        assert "zone 1" in code(lambda: s.central_bracket())
    with _solver(gpu_lib, zones, T) as s:
        code(lambda: s.central_bracket())                          # no homes
        s.set_homes(**hm)
        code(lambda: s.central_bracket())                          # no tariff
        s.set_tariff(cost)
        code(lambda: s.network_check("central"))                   # no bracket yet
        code(lambda: s.central_bracket(iters=-1))
        code(lambda: s.central_bracket(vset=1.05, vhigh=1.05))
        code(lambda: s.central_bracket(vset=1.06, vhigh=1.05))
        code(lambda: s.central_bracket(row_tol=-1e-9))
        code(lambda: s.central_bracket(row_tol=float("nan")))
        mask = np.empty((s.H, 2), dtype=np.uint64)
        rc = s.lib.revs_central_bracket(s._h, 1.0, 1.05, 1e-9, 10, None,
                                        mask.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), 2, None, None)
        assert rc == 1
        s.central_bracket(iters=5)
        s.network_check("central")
        s.set_tariff(cost)
        code(lambda: s.network_check("central"))                   # new inputs invalidate the kept schedule
        bad = {k: np.array(v, copy=True) for k, v in hm.items()}
        h = int(np.nonzero(bad["has_ev"])[0][0])
        bad["end"][h] = bad["start"][h] + 1
        bad["capacity"][h] = bad["rating"][h] * 2.5 / (0.9 - bad["initial"][h])     # n_min = 3 > 1 window hour
        s.set_homes(**bad)
        code(lambda: s.central_bracket(iters=5), c=3)
        s.set_homes(**hm)
        s.central_bracket(iters=5)                                 # the solver still works
        s.network_check("central")

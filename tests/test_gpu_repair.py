"""GPU: the greedy voltage repair (revs_repair_schedule) against the numpy model of tests/repair_ref.py, on mixed
zones, on reference-shaped feeders with the bench's ADMM parameters and on a tree-only zone; pipelines,
determinism, side effects and argument errors."""
import ctypes

import numpy as np
import pytest

import network_ref as NR
import repair_ref as RR
from revs_admm_b200.feeder import population, radial_feeder, synthetic_homes, synthetic_tariff
from test_gpu_network import BENCH, _mixed_zones, _solved, _solver

pytestmark = pytest.mark.gpu

LOOSE = dict(kappa=5.0, iter_max=4, vset=1.0, vlow=0.95, vhigh=1.05)


def _vhigh(zones, hm, factor):
    """vhigh (vset = 1) whose limit is `factor` times the largest drop of the base load alone: the homes' chargers,
    scheduled under LOOSE limits, violate it."""
    return float(np.sqrt(1.0 + factor * NR.network_check(zones, hm["load"])["drop"].max()))


def _model(s, zones, hm, cost, vset, vhigh, row_tol=1e-9):
    r = s.results(want_diff=False)
    return RR.repair(zones, r["P_sch"], r["P_ev"] > 0.0, hm, cost, vset=vset, vhigh=vhigh, row_tol=row_tol)


def _check_equal(got, ref, T):
    assert np.array_equal(got["zone_info"], ref["zone_info"])
    assert np.array_equal(RR.unpack(got["mask"], T), ref["bits"])
    assert np.array_equal(got["P_sch"], ref["P_sch"])


@pytest.mark.parametrize("T", [24, 37, 96])
def test_matches_model_on_mixed_zones(gpu_lib, T):
    zones = _mixed_zones(T)
    hm = synthetic_homes(sum(z.n_res for z in zones), T, seed=T)
    cost = synthetic_tariff(T)
    vhigh = _vhigh(zones, hm, 1.3)
    with _solved(gpu_lib, zones, hm, cost, T, **LOOSE) as s:
        got = s.repair_schedule(vset=1.0, vhigh=vhigh, mask=True)
        ref = _model(s, zones, hm, cost, 1.0, vhigh)
    _check_equal(got, ref, T)
    assert got["zones_violated"] > 0 and got["moves"] + got["drops"] > 0


def _refshape(n):
    trees, hm, cost, sizes, T = population("refshape", n, seed=0)
    return trees, hm, cost, T


def test_reference_shaped_feeders(gpu_lib):
    import bench
    trees, hm, cost, T = _refshape(3)
    kw = dict(vset=BENCH["vset"], vhigh=BENCH["vhigh"])
    with _solved(gpu_lib, trees, hm, cost, T, **BENCH) as s:
        before = s.network_check("schedule", zones=True, **kw)
        got = s.repair_schedule(mask=True, **kw)
        after = s.network_check("repaired", zones=True, **kw)
        ref = _model(s, trees, hm, cost, **kw)
        P0 = s.results(want_diff=False)["P_sch"]
    _check_equal(got, ref, T)
    assert before["summary"]["rows_violated"] > 0 and got["zones_violated"] > 0
    st = got["zone_info"][:, 0]
    assert (after["zone_worst"][st <= 1, 1] <= 1e-9).all()
    assert (after["zone_worst"][st == 2, 1] <= before["zone_worst"][st == 2, 1]).all()
    if got["zones_left"] == 0:
        assert after["summary"]["rows_violated"] == 0
    _, lb, _ = bench.objective_check(trees, hm, cost, P0, T)
    assert float((got["P_sch"] @ cost).sum()) >= lb


def test_tree_only_zone_uses_the_global_state(gpu_lib):
    T = 96
    zones = [radial_feeder(2300, seed=3, r_scale=0.07)]
    hm = synthetic_homes(2300, T, seed=4)
    cost = synthetic_tariff(T)
    vhigh = _vhigh(zones, hm, 1.3)
    with _solved(gpu_lib, zones, hm, cost, T, **LOOSE) as s:
        got = s.repair_schedule(vset=1.0, vhigh=vhigh, mask=True)
        ref = _model(s, zones, hm, cost, 1.0, vhigh)
    _check_equal(got, ref, T)
    assert got["zones_violated"] == 1


def test_pipelines_equal_one_solver(gpu_lib):
    trees, hm, cost, T = _refshape(6)
    kw = dict(vset=BENCH["vset"], vhigh=BENCH["vhigh"], mask=True)
    with _solved(gpu_lib, trees, hm, cost, T, **BENCH) as a:
        ra = a.repair_schedule(**kw)
        na = a.network_check("repaired", vset=BENCH["vset"], zones=True)
    with _solved(gpu_lib, trees, hm, cost, T, cls=lambda sizes, T: gpu_lib.PipelinedSolver(sizes, T, pipelines=4),
                 **BENCH) as b:
        assert len(b.parts) == 4
        rb = b.repair_schedule(**kw)
        nb = b.network_check("repaired", vset=BENCH["vset"], zones=True)
    for k in ("P_sch", "mask", "zone_info"):
        assert np.array_equal(ra[k], rb[k]), k
    for k in ("moves", "drops", "zones_violated", "zones_repaired", "zones_left"):
        assert ra[k] == rb[k], k
    assert na["summary"] == nb["summary"] and np.array_equal(na["zone_worst"], nb["zone_worst"])


def test_deterministic_and_without_side_effects(gpu_lib):
    trees, hm, cost, T = _refshape(2)
    kw = dict(vset=BENCH["vset"], vhigh=BENCH["vhigh"], mask=True)
    with _solved(gpu_lib, trees, hm, cost, T, **BENCH) as s:
        before, est = s.results(), s.estimate()
        chk = s.network_check("schedule", vset=BENCH["vset"], full=True, zones=True)
        n0 = s.stats()["kernel_launches"]
        a = s.repair_schedule(**kw)
        assert s.stats()["kernel_launches"] > n0
        b = s.repair_schedule(**kw)
        for k in ("P_sch", "mask", "zone_info"):
            assert a[k].tobytes() == b[k].tobytes(), k
        after, est2 = s.results(), s.estimate()
        for k in before:
            assert np.array_equal(before[k], after[k]), k
        assert all(np.array_equal(x, y) for x, y in zip(est, est2))
        chk2 = s.network_check("schedule", vset=BENCH["vset"], full=True, zones=True)
        assert chk["summary"] == chk2["summary"]
        for k in ("voltage", "loading", "zone_worst"):
            assert np.array_equal(chk[k], chk2[k]), k
        s.solve_admm(**BENCH)
        again = s.results()
        for k in before:
            assert np.array_equal(before[k], again[k]), k


def test_argument_errors(gpu_lib):
    T = 24
    zones = _mixed_zones(1)[:2]
    hm = synthetic_homes(sum(z.n_res for z in zones), T, seed=2)

    def code(fn):
        with pytest.raises(gpu_lib.RevsError) as e:
            fn()
        assert e.value.code == 1, str(e.value)
        return str(e.value)

    lib = gpu_lib._cabi.load()
    assert lib.revs_repair_schedule(None, 1.0, 1.05, 1e-9, None, None, 1, None) == 1
    with gpu_lib.Solver([z.n_res for z in zones], T) as s:
        s.set_feeder_tree(0, zones[0].parent, zones[0].r, zones[0].res_node)
        s.set_sensitivity(1, np.eye(zones[1].n_res) * 1e-3)
        s.set_homes(**hm)
        s.set_tariff(synthetic_tariff(T))
        s.solve_admm(iter_max=2)
        assert "zone 1" in code(lambda: s.repair_schedule())
    with _solver(gpu_lib, zones, T) as s:
        s.set_homes(**hm)
        s.set_tariff(synthetic_tariff(T))
        code(lambda: s.repair_schedule())                          # no ADMM iteration
        s.solve_admm(iter_max=2)
        code(lambda: s.network_check("repaired"))                  # no repair of this run
        code(lambda: s.repair_schedule(vset=1.05, vhigh=1.05))
        code(lambda: s.repair_schedule(vset=1.06, vhigh=1.05))
        code(lambda: s.repair_schedule(row_tol=-1e-9))
        code(lambda: s.repair_schedule(row_tol=float("nan")))
        mask = np.empty((s.H, 2), dtype=np.uint64)
        rc = s.lib.revs_repair_schedule(s._h, 1.0, 1.05, 1e-9, None, mask.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)),
                                        2, None)
        assert rc == 1
        s.repair_schedule()
        s.network_check("repaired")
        s.solve_admm(iter_max=2)
        code(lambda: s.network_check("repaired"))                  # a new run invalidates the repair
        s.repair_schedule()                                        # the solver still works

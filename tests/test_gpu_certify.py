"""GPU: the certificate of voltage infeasibility (revs_certify_infeasible) against the numpy model of
tests/certify_ref.py, on mixed zones, per-home windows, reference-shaped feeders at the bench's limits and a tree-only
zone; consistency with central_bracket, pipelines, determinism, side effects and argument errors."""
import ctypes

import numpy as np
import pytest

import certify_ref as CF
import network_ref as NR
from revs_admm_b200.feeder import population, radial_feeder, synthetic_homes
from test_central_model import _homes
from test_gpu_network import BENCH, _mixed_zones, _solver

pytestmark = pytest.mark.gpu

LIMITS = dict(vset=BENCH["vset"], vhigh=BENCH["vhigh"])


def _vhigh(zones, hm, factor):
    """vhigh (vset = 1) whose limit is `factor` times the largest drop of the base load alone."""
    return float(np.sqrt(1.0 + factor * NR.network_check(zones, hm["load"])["drop"].max()))


def _ready(lib, zones, hm, T, cost=None, cls=None):
    s = _solver(lib, zones, T, cls=cls)
    s.set_homes(**hm)
    if cost is not None:
        s.set_tariff(cost)
    return s


def _check(lib, zones, hm, T, **kw):
    with _ready(lib, zones, hm, T) as s:
        got = s.certify_infeasible(**kw)
    ref = CF.certify(zones, hm, **kw)
    assert np.array_equal(got["zone_cert"], ref["zone_cert"])
    return got


@pytest.mark.parametrize("T", [24, 37, 96])
def test_matches_model_on_mixed_zones(gpu_lib, T):
    zones = _mixed_zones(T)
    hm = synthetic_homes(sum(z.n_res for z in zones), T, seed=T)
    kinds = set()
    for factor in (0.9, 1.1, 1.4, 2.0):
        got = _check(gpu_lib, zones, hm, T, vset=1.0, vhigh=_vhigh(zones, hm, factor))
        kinds |= set(got["zone_cert"][:, 0].tolist())
    assert kinds == {0, 1, 2}


@pytest.mark.parametrize("T", [24, 96])
def test_matches_model_with_per_home_windows(gpu_lib, T):
    zones = _mixed_zones(T + 1)
    hm = _homes(sum(z.n_res for z in zones), T, seed=T + 1)
    kinds = set()
    for factor in (1.1, 1.5, 2.5):
        got = _check(gpu_lib, zones, hm, T, vset=1.0, vhigh=_vhigh(zones, hm, factor))
        kinds |= set(got["zone_cert"][:, 0].tolist())
    assert 2 in kinds


def test_reference_shaped_feeders(gpu_lib):
    trees, hm, cost, sizes, T = population("refshape", 3, seed=0)
    got = _check(gpu_lib, trees, hm, T, **LIMITS)
    assert got["zone_cert"][6].tolist() == [2, 121, 4, 10]
    assert got["certified"] == sum(got["zones_kind"][1:]) >= 1


def test_tree_only_zone(gpu_lib):
    T = 96
    zones = [radial_feeder(2300, seed=3, r_scale=0.07)]
    hm = synthetic_homes(2300, T, seed=4)
    kinds = [_check(gpu_lib, zones, hm, T, vset=1.0, vhigh=_vhigh(zones, hm, f))["zone_cert"][0, 0] for f in (0.95, 1.3)]
    assert kinds == [1, 2]


def test_consistent_with_the_bracket(gpu_lib):
    """No zone with a voltage-feasible schedule (bracket status 0 or 1) is certified; central_status takes the rest."""
    trees, hm, cost, sizes, T = population("refshape", 3, seed=0)
    with _ready(gpu_lib, trees, hm, T, cost) as s:
        br = s.central_bracket(iters=30, **LIMITS)
        cert = s.certify_infeasible(**LIMITS)
    st = gpu_lib.central_status(br["zone_info"], cert["zone_cert"])
    assert ((st == 3) == ((br["zone_info"][:, 0] == 3) | (cert["zone_cert"][:, 0] > 0))).all()
    assert st[6] == 3 and br["zone_info"][6, 0] == 2


def test_pipelines_equal_one_solver(gpu_lib):
    trees, hm, cost, sizes, T = population("refshape", 6, seed=0)
    with _ready(gpu_lib, trees, hm, T) as a:
        ra = a.certify_infeasible(**LIMITS)
    with _ready(gpu_lib, trees, hm, T, cls=lambda sizes, T: gpu_lib.PipelinedSolver(sizes, T, pipelines=4)) as b:
        assert len(b.parts) == 4
        rb = b.certify_infeasible(**LIMITS)
    assert ra["zone_cert"].tobytes() == rb["zone_cert"].tobytes()
    assert ra["zones_kind"] == rb["zones_kind"] and ra["certified"] == rb["certified"]


def test_deterministic_and_changes_no_state(gpu_lib):
    trees, hm, cost, sizes, T = population("refshape", 2, seed=0)
    with _ready(gpu_lib, trees, hm, T, cost) as s:
        s.solve_admm(**BENCH)
        before = s.results()
        rep = s.repair_schedule(**LIMITS)
        chk_r = s.network_check("repaired", zones=True, **LIMITS)
        br = s.central_bracket(iters=10, mask=True, **LIMITS)
        chk_c = s.network_check("central", zones=True, **LIMITS)
        n0 = s.stats()["kernel_launches"]
        a = s.certify_infeasible(**LIMITS)
        assert s.stats()["kernel_launches"] > n0
        b = s.certify_infeasible(**LIMITS)
        assert a["zone_cert"].tobytes() == b["zone_cert"].tobytes()
        after = s.results()
        for k in before:
            assert np.array_equal(before[k], after[k]), k
        c = s.network_check("central", zones=True, **LIMITS)
        assert c["summary"] == chk_c["summary"] and np.array_equal(c["zone_worst"], chk_c["zone_worst"])
        r = s.network_check("repaired", zones=True, **LIMITS)
        assert r["summary"] == chk_r["summary"] and np.array_equal(r["zone_worst"], chk_r["zone_worst"])
        br2 = s.central_bracket(iters=10, mask=True, **LIMITS)
        for k in ("P_sch", "mask", "zone_bounds", "zone_info"):
            assert np.array_equal(br[k], br2[k]), k
        assert np.array_equal(rep["P_sch"], s.repair_schedule(**LIMITS)["P_sch"])


def test_argument_errors(gpu_lib):
    T = 24
    zones = _mixed_zones(1)[:2]
    hm = synthetic_homes(sum(z.n_res for z in zones), T, seed=2)

    def code(fn, c=1):
        with pytest.raises(gpu_lib.RevsError) as e:
            fn()
        assert e.value.code == c, str(e.value)
        return str(e.value)

    lib = gpu_lib._cabi.load()
    assert lib.revs_certify_infeasible(None, 1.0, 1.05, 1e-9, None, None) == 1
    with gpu_lib.Solver([z.n_res for z in zones], T) as s:
        s.set_feeder_tree(0, zones[0].parent, zones[0].r, zones[0].res_node)
        s.set_sensitivity(1, np.eye(zones[1].n_res) * 1e-3)
        s.set_homes(**hm)
        assert "zone 1" in code(lambda: s.certify_infeasible(1.0, 1.05))
    with _solver(gpu_lib, zones, T) as s:
        code(lambda: s.certify_infeasible(1.0, 1.05))              # no homes
        s.set_homes(**hm)
        code(lambda: s.certify_infeasible(1.05, 1.05))
        code(lambda: s.certify_infeasible(1.06, 1.05))
        code(lambda: s.certify_infeasible(1.0, 1.05, row_tol=-1e-9))
        code(lambda: s.certify_infeasible(1.0, 1.05, row_tol=float("nan")))
        vh = _vhigh(zones, hm, 1.2)
        ref = CF.certify(zones, hm, vset=1.0, vhigh=vh)["zone_cert"]
        n = ctypes.c_int(-1)
        assert s.lib.revs_certify_infeasible(s._h, 1.0, vh, 1e-9, None, ctypes.byref(n)) == 0
        assert n.value == int((ref[:, 0] > 0).sum())
        bad = {k: np.array(v, copy=True) for k, v in hm.items()}
        h = int(np.nonzero(bad["has_ev"])[0][0])
        bad["rating"][h] = np.inf
        s.set_homes(**bad)
        assert "rating" in code(lambda: s.certify_infeasible(1.0, 1.05))
        bad = {k: np.array(v, copy=True) for k, v in hm.items()}
        bad["end"][h] = bad["start"][h] + 1
        bad["capacity"][h] = bad["rating"][h] * 2.5 / (0.9 - bad["initial"][h])     # n_min = 3 > 1 window hour
        s.set_homes(**bad)
        code(lambda: s.certify_infeasible(1.0, 1.05), c=3)
        s.set_homes(**hm)
        assert np.array_equal(s.certify_infeasible(1.0, vh)["zone_cert"], ref)      # the solver still works

"""GPU: the hosting capacity (revs_hosting_capacity) against the numpy model of tests/hosting_ref.py, bit for bit, on
mixed zones, per-home windows, reference-shaped feeders, feeder 121144 with its line ratings, a tree-only zone and the
zones of the global-scratch path; sources, the certificate's base-load zones, pipelines, determinism, side effects and
argument errors."""
import ctypes

import numpy as np
import pytest

import hosting_ref as HR
import network_ref as NR
from revs_admm_b200.feeder import population, radial_feeder, synthetic_feeder, synthetic_homes
from test_central_model import _homes
from test_gpu_network import BENCH, _mixed_zones, _solved, _solver

pytestmark = pytest.mark.gpu

LIMITS = dict(vset=BENCH["vset"], vhigh=BENCH["vhigh"])


def _scale(n, seed):
    rng = np.random.default_rng(seed)
    s = rng.choice([-1.0, 1.0], n) / rng.uniform(5.0, 80.0, n)
    s[rng.random(n) < 0.3] = 0.0
    return s


def _same(got, ref):
    assert np.array_equal(got["home_cap"], ref["home_cap"])
    assert np.array_equal(got["zone_uniform"], ref["zone_uniform"])
    assert np.array_equal(got["zone_counts"], ref["zone_counts"])


@pytest.mark.parametrize("T", [24, 37, 96])
def test_matches_model_on_mixed_zones(gpu_lib, T):
    zones = _mixed_zones(T)
    H, N = sum(z.n_res for z in zones), sum(z.n_nodes for z in zones)
    hm = synthetic_homes(H, T, seed=T)
    rng = np.random.default_rng(T)
    with _solver(gpu_lib, zones, T) as s:
        s.set_homes(**hm)
        for hi, scale in ((2.0, None), (2.0, _scale(N, T)), (30.0, None), (30.0, _scale(N, T + 1))):
            P = rng.uniform(0.0, hi, (H, T))
            kw = dict(vset=1.0, vhigh=1.04, row_tol=1e-9, scale=scale)
            got = s.hosting_capacity(P, **kw)
            _same(got, HR.hosting(zones, P, hm=hm, **kw))
            assert got["window_steps"] == int(got["zone_counts"][:, 0].sum()) > 0
            if scale is not None:
                assert got["thermal_bound"] > 0


@pytest.mark.parametrize("T", [24, 96])
def test_matches_model_with_per_home_windows(gpu_lib, T):
    zones = _mixed_zones(T + 1)
    hm = _homes(sum(z.n_res for z in zones), T, seed=T + 1)
    with _solver(gpu_lib, zones, T) as s:
        s.set_homes(**hm)
        got = s.hosting_capacity(hm["load"] * 3.0, vset=1.0, vhigh=1.03)
    ref = HR.hosting(zones, hm["load"] * 3.0, vset=1.0, vhigh=1.03, hm=hm)
    _same(got, ref)
    assert 0 < got["window_steps_open"] < got["window_steps"]


def test_reference_shaped_feeders(gpu_lib):
    trees, hm, cost, sizes, T = population("refshape", 3, seed=0)
    scale = _scale(sum(t.n_nodes for t in trees), 3) * 0.2
    with _solver(gpu_lib, trees, T) as s:
        s.set_homes(**hm)
        for sc in (None, scale):
            got = s.hosting_capacity(hm["load"] * 2.0, scale=sc, **LIMITS)
            _same(got, HR.hosting(trees, hm["load"] * 2.0, scale=sc, hm=hm, **LIMITS))
    m = got["home_cap_min"]
    assert m["value"] == got["home_cap"].min()
    assert got["home_cap"][sum(sizes[:m["zone"]]) + m["index"], m["step"]] == m["value"]


def test_reference_feeder_with_line_ratings(gpu_lib, case121144):
    from revs_admm_b200 import lpsolver
    dist, homes = case121144["dist"], case121144["homes"]
    tree, zones, perm = lpsolver._zones(dist)
    res = tree.res_ids
    P = np.array([np.asarray(homes[res[j]]["LOAD"], dtype=np.float64) * 3.0 for j in perm])
    T = P.shape[1]
    zt = [z for z, _ in zones]
    scale = np.concatenate([z.edge_sign / np.array([np.sqrt(3) * lpsolver.LINE_RATING_KVA[t] for t in z.edge_type])
                            for z in zt])
    with _solver(gpu_lib, zt, T) as s:
        got = s.hosting_capacity(P, scale=scale, **LIMITS)
        free = s.hosting_capacity(P, **LIMITS)
    _same(got, HR.hosting(zt, P, scale=scale, **LIMITS))
    _same(free, HR.hosting(zt, P, **LIMITS))
    assert (got["home_cap"] <= free["home_cap"]).all()


def test_tree_only_and_global_scratch_zones(gpu_lib):
    """The 2,300-residence tree-only zone, the zones of test_large_zones (shared memory of both classes and the global
    scratch of a zone above the shared-memory size), next to a small zone."""
    T = 96
    zones = [radial_feeder(n, seed=n, r_scale=0.07) for n in (2300, 10000, 15000, 25000)] + [synthetic_feeder(40, seed=1)]
    H, N = sum(z.n_res for z in zones), sum(z.n_nodes for z in zones)
    P = np.random.default_rng(0).uniform(0.0, 3.0, (H, T))
    scale = _scale(N, 9) * 0.05
    with _solver(gpu_lib, zones, T) as s:
        got = s.hosting_capacity(P, vset=1.03, vhigh=1.05, scale=scale)
    ref = HR.hosting(zones, P, vset=1.03, vhigh=1.05, scale=scale)
    _same(got, ref)
    assert np.isfinite(got["home_cap"]).all() and (got["home_cap"] > 0.0).any()


def test_sources_agree(gpu_lib):
    trees, hm, cost, sizes, T = population("refshape", 2, seed=0)
    with _solved(gpu_lib, trees, hm, cost, T, **BENCH) as s:
        rep = s.repair_schedule(**LIMITS)["P_sch"]
        cen = s.central_bracket(iters=10, **LIMITS)["P_sch"]
        for src, P in (("schedule", s.results()["P_sch"]), ("estimate", s.estimate()[0]), ("repaired", rep),
                       ("central", cen)):
            a = s.hosting_capacity(src, **LIMITS)
            b = s.hosting_capacity(P, **LIMITS)
            for k in ("home_cap", "zone_uniform", "zone_counts"):
                assert a[k].tobytes() == b[k].tobytes(), (src, k)


def test_base_load_certificate_zones_have_no_capacity(gpu_lib):
    """Kind-1 zones of certify_infeasible (the base load alone violates a row): with P = load, every home whose
    R[witness, h] > 0 has capacity 0 at the witness step."""
    T = 96
    zones = [radial_feeder(2300, seed=3, r_scale=0.07)] + _mixed_zones(T)
    hm = synthetic_homes(sum(z.n_res for z in zones), T, seed=4)
    vh = float(np.sqrt(1.0 + 0.95 * NR.network_check(zones, hm["load"])["drop"].max()))
    with _solver(gpu_lib, zones, T) as s:
        s.set_homes(**hm)
        cert = s.certify_infeasible(1.0, vh)["zone_cert"]
        cap = s.hosting_capacity(hm["load"], vset=1.0, vhigh=vh)["home_cap"]
    off = np.concatenate([[0], np.cumsum([z.n_res for z in zones])])
    kind1 = np.nonzero(cert[:, 0] == 1)[0]
    assert len(kind1) > 0
    for z in kind1:
        i, t = int(cert[z, 1]), int(cert[z, 2])
        c = HR.RR._Columns(zones[z])
        reach = np.array([c(h)[i] > 0.0 for h in range(zones[z].n_res)])
        assert reach.any() and (cap[off[z]:off[z + 1]][reach, t] == 0.0).all()


def test_pipelines_equal_one_solver(gpu_lib):
    trees, hm, cost, sizes, T = population("refshape", 6, seed=0)
    scale = _scale(sum(t.n_nodes for t in trees), 1) * 0.2
    res = []
    for cls in (None, lambda sizes, T: gpu_lib.PipelinedSolver(sizes, T, pipelines=4)):
        with _solved(gpu_lib, trees, hm, cost, T, cls=cls, **BENCH) as s:
            res.append([s.hosting_capacity(src, scale=scale, **LIMITS) for src in ("schedule", hm["load"] * 2.0)])
    for a, b in zip(*res):
        for k in ("home_cap", "zone_uniform", "zone_counts"):
            assert a[k].tobytes() == b[k].tobytes(), k
        for k in ("window_steps", "window_steps_open", "thermal_bound", "home_cap_min", "uniform_min"):
            assert a[k] == b[k], k


def test_deterministic_and_changes_no_state(gpu_lib):
    trees, hm, cost, sizes, T = population("refshape", 2, seed=0)
    scale = _scale(sum(t.n_nodes for t in trees), 2) * 0.2
    with _solved(gpu_lib, trees, hm, cost, T, **BENCH) as s:
        before, est = s.results(), s.estimate()
        s.repair_schedule(**LIMITS)
        s.central_bracket(iters=10, **LIMITS)
        checks = {src: s.network_check(src, full=True, zones=True, **LIMITS)
                  for src in ("schedule", "estimate", "repaired", "central")}
        n0 = s.stats()["kernel_launches"]
        a = s.hosting_capacity("schedule", scale=scale, **LIMITS)
        assert s.stats()["kernel_launches"] > n0
        b = s.hosting_capacity("schedule", scale=scale, **LIMITS)
        for k in ("home_cap", "zone_uniform", "zone_counts"):
            assert a[k].tobytes() == b[k].tobytes(), k
        only = s.hosting_capacity("schedule", scale=scale, homes=False, uniform=False, **LIMITS)
        assert only["home_cap"] is None and np.array_equal(only["zone_counts"], a["zone_counts"])
        after, est2 = s.results(), s.estimate()
        for k in before:
            assert np.array_equal(before[k], after[k]), k
        assert all(x.tobytes() == y.tobytes() for x, y in zip(est, est2))
        for src, c in checks.items():
            d = s.network_check(src, full=True, zones=True, **LIMITS)
            assert d["summary"] == c["summary"], src
            for k in ("voltage", "loading", "zone_worst"):
                assert d[k].tobytes() == c[k].tobytes(), (src, k)


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
    assert lib.revs_hosting_capacity(None, 2, None, 1.0, 1.05, 1e-9, None, None, None, None) == 1
    with gpu_lib.Solver([z.n_res for z in zones], T) as s:
        s.set_feeder_tree(0, zones[0].parent, zones[0].r, zones[0].res_node)
        s.set_sensitivity(1, np.eye(zones[1].n_res) * 1e-3)
        assert "zone 1" in code(lambda: s.hosting_capacity(np.zeros((s.H, T))))
    with _solver(gpu_lib, zones, T) as s:
        s.set_homes(**hm)
        P = hm["load"]
        code(lambda: s.hosting_capacity("schedule"))
        code(lambda: s.hosting_capacity("estimate"))
        code(lambda: s.hosting_capacity("repaired"))
        code(lambda: s.hosting_capacity("central"))
        code(lambda: s.hosting_capacity(P, vset=1.05, vhigh=1.05))
        code(lambda: s.hosting_capacity(P, vset=1.06, vhigh=1.05))
        code(lambda: s.hosting_capacity(P, row_tol=-1e-9))
        code(lambda: s.hosting_capacity(P, row_tol=float("nan")))
        bad = np.zeros(s.total_nodes)
        for v in (np.nan, np.inf):
            bad[3] = v
            assert "scale" in code(lambda: s.hosting_capacity(P, scale=bad))
        for src, p in ((gpu_lib.REVS_NET_HOST, None), (7, P.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))):
            assert s.lib.revs_hosting_capacity(s._h, src, p, 1.0, 1.05, 1e-9, None, None, None, None) == 1
        got = s.hosting_capacity(P, vset=1.0, vhigh=1.05)                   # the solver still works
        _same(got, HR.hosting(zones, P, vset=1.0, vhigh=1.05, hm=hm))

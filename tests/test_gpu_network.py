"""GPU: the population network check (revs_network_check) against revs_reliability, the numpy model, the reference
feeder's compute_voltage / compute_flows, the ADMM certificate and the bench's host check; pipelines, determinism,
side effects and argument errors."""
import ctypes

import numpy as np
import pytest

import network_ref as NR
from revs_admm_b200.feeder import FeederTree, population, radial_feeder, synthetic_feeder, synthetic_homes, synthetic_tariff

pytestmark = pytest.mark.gpu

BENCH = dict(kappa=5.0, iter_max=15, vset=1.03, vlow=0.95, vhigh=1.05)      # bench.py ADMM


def _mixed_zones(seed):
    """Zones with several residences on one node and nodes without any, plus a one-node zone."""
    rng = np.random.default_rng(seed)
    out = []
    for n in (40, 75, 130):
        t = synthetic_feeder(n, seed=seed + n, laterals=3, r_secondary=3e-4)
        res = t.res_node.copy()
        res[1::4] = res[0]
        res[2::7] = rng.integers(0, t.n_nodes - n, len(res[2::7]))
        out.append(FeederTree(parent=t.parent, r=t.r, res_node=res.astype(np.int32)))
    out.insert(1, FeederTree(parent=np.array([-1], np.int32), r=np.array([1e-3]), res_node=np.zeros(3, np.int32)))
    return out


def _solver(lib, zones, T, one_by_one=False, cls=None):
    s = (cls or lib.Solver)([z.n_res for z in zones], T)
    if one_by_one:
        for f, z in enumerate(zones):
            s.set_feeder_tree(f, z.parent, z.r, z.res_node)
    else:
        s.set_feeder_trees(zones)
    return s


def _solved(lib, zones, hm, cost, T, cls=None, **kw):
    s = _solver(lib, zones, T, cls=cls)
    s.set_homes(**hm)
    s.set_tariff(cost)
    s.solve_admm(**kw)
    return s


@pytest.mark.parametrize("T", [24, 37, 96])
@pytest.mark.parametrize("one_by_one", [False, True])
def test_matches_reliability_and_model(gpu_lib, T, one_by_one):
    zones = _mixed_zones(T)
    rng = np.random.default_rng(T)
    H, N = sum(z.n_res for z in zones), sum(z.n_nodes for z in zones)
    P = rng.uniform(0.0, 2.0, (H, T))
    scale = rng.choice([-1.0, 1.0], N) / rng.uniform(20.0, 200.0, N)
    kw = dict(vset=1.03, vlow=0.97, vhigh=1.04, row_tol=1e-9)
    with _solver(gpu_lib, zones, T, one_by_one) as s:
        got = s.network_check(P, scale=scale, full=True, zones=True, **kw)
        ref = NR.network_check(zones, P, scale=scale, **kw)
        off = noff = 0
        for f, z in enumerate(zones):
            rows = np.arange(z.n_nodes)
            Pz = P[off:off + z.n_res]
            volt = s.reliability(f, gpu_lib.REVS_REL_VOLTAGE, rows, vset=kw["vset"], P=Pz)
            flow = s.reliability(f, gpu_lib.REVS_REL_FLOW, rows, scale=scale[noff:noff + z.n_nodes], P=Pz)
            assert np.abs(got["voltage"][noff:noff + z.n_nodes] - volt).max() <= 1e-12
            assert np.abs(got["loading"][noff:noff + z.n_nodes] - flow).max() <= 1e-12 * np.abs(flow).max()
            off += z.n_res
            noff += z.n_nodes
    # the kernel sums in the model's order: identical outputs, and the summary is the reduction of those outputs
    assert np.array_equal(got["voltage"], ref["voltage"])
    assert np.array_equal(got["loading"], ref["loading"])
    assert got["summary"] == ref["summary"]
    assert np.array_equal(got["zone_worst"], ref["zone_worst"])


def test_summary_is_the_reduction_of_the_arrays(gpu_lib):
    """Exact ties (a repeated zone, repeated steps, a zone without load) go to the lowest (zone, index, step)."""
    T = 24
    base = _mixed_zones(3)
    zones = [base[0], base[0], base[1], base[2]]
    rng = np.random.default_rng(5)
    P0 = rng.uniform(0.0, 3.0, (base[0].n_res, T))
    P0[:, 5] = P0[:, 4]
    P = np.concatenate([P0, P0, np.zeros((base[1].n_res, T)), rng.uniform(0.0, 0.2, (base[2].n_res, T))])
    kw = dict(vset=1.0, vlow=0.98, vhigh=1.01, row_tol=1e-9)
    with _solver(gpu_lib, zones, T) as s:
        got = s.network_check(P, full=True, zones=True, **kw)
        summary_only = s.network_check(P, **kw)
    ref = NR.network_check(zones, P, **kw)
    assert np.array_equal(np.sqrt(1.0 - ref["drop"]), got["voltage"])      # the model's drops are the kernel's
    D = [ref["drop"][a:b] for a, b in _blocks(zones)]
    L = [got["loading"][a:b] for a, b in _blocks(zones)]
    summary, zw = NR.summarize(zones, D, L, scaled=False, **kw)
    assert got["summary"] == summary == summary_only["summary"]
    assert np.array_equal(got["zone_worst"], zw)
    assert summary["drop_zone"] == 0 and summary["loading_zone"] == 0
    assert summary_only["voltage"] is None and summary_only["zone_worst"] is None


def _blocks(zones):
    off = np.concatenate([[0], np.cumsum([z.n_nodes for z in zones])])
    return list(zip(off[:-1], off[1:]))


def test_reference_feeder_matches_compute_voltage_and_flows(gpu_lib, case121144):
    from revs_admm_b200 import lpsolver
    dist, homes = case121144["dist"], case121144["homes"]
    tree, zones, perm = lpsolver._zones(dist)
    res = tree.res_ids
    p = {h: np.asarray(homes[h]["LOAD"], dtype=np.float64) * 3.0 for h in res}
    T = len(p[res[0]])
    P = np.array([p[res[j]] for j in perm])
    zt = [z for z, _ in zones]
    scale = np.concatenate([z.edge_sign / np.array([np.sqrt(3) * lpsolver.LINE_RATING_KVA[t] for t in z.edge_type])
                            for z in zt])
    with _solver(gpu_lib, zt, T) as s:
        volt = s.network_check(P, vset=1.03, full=True)["voltage"]
        load = s.network_check(P, scale=scale, full=True)["loading"]
    v_ref = lpsolver.compute_voltage(dist, p, vset=1.03)
    f_ref = lpsolver.compute_flows(dist, p)
    fmax = max(np.abs(v).max() for v in f_ref.values())
    for (a, _), z in zip(_blocks(zt), zt):
        for i, n in enumerate(z.node_ids):
            assert np.abs(volt[a + i] - np.asarray(v_ref[n])).max() <= 1e-12
            assert np.abs(load[a + i] - np.asarray(f_ref[z.edge_keys[i]])).max() <= 1e-12 * fmax


def _refshape(n_feeders):
    trees, hm, cost, sizes, T = population("refshape", n_feeders, seed=0)
    return trees, hm, cost, T


def test_sources_agree(gpu_lib):
    trees, hm, cost, T = _refshape(2)
    with _solved(gpu_lib, trees, hm, cost, T, **BENCH) as s:
        for src, P in (("schedule", s.results()["P_sch"]), ("estimate", s.estimate()[0])):
            a = s.network_check(src, vset=1.03, full=True, zones=True)
            b = s.network_check(P, vset=1.03, full=True, zones=True)
            assert a["summary"] == b["summary"]
            for k in ("voltage", "loading", "zone_worst"):
                assert np.array_equal(a[k], b[k]), (src, k)


def test_estimate_satisfies_the_voltage_rows(gpu_lib):
    """The operator's estimate satisfies its voltage rows (KKT certificate), on every zone of the population."""
    trees, hm, cost, T = _refshape(4)
    with _solved(gpu_lib, trees, hm, cost, T, **BENCH) as s:
        c = s.network_check("estimate", vset=1.03, vlow=0.95, vhigh=1.05)["summary"]
    assert c["row_excess_max"] <= 1e-9 and c["rows_violated"] == 0
    trees, hm, cost, sizes, T = population("radial10k", 1, seed=0)
    with _solved(gpu_lib, trees, hm, cost, T, **BENCH) as s:
        c = s.network_check("estimate", vset=1.03, vlow=0.95, vhigh=1.05)["summary"]
    assert c["row_excess_max"] <= 1e-9 and c["rows_violated"] == 0


def test_matches_the_bench_host_check(gpu_lib):
    trees, hm, cost, T = _refshape(16)
    assert len(trees) >= 64
    with _solved(gpu_lib, trees, hm, cost, T, **BENCH) as s:
        P = s.results()["P_sch"]
        zw = s.network_check("schedule", vset=1.03, vlow=0.95, vhigh=1.05, zones=True)["zone_worst"]
    u = BENCH["vhigh"] ** 2 - BENCH["vset"] ** 2
    off = np.concatenate([[0], np.cumsum([t.n_res for t in trees])])
    host = np.array([(tr.drop(P[off[z]:off[z + 1]]) - u).max() for z, tr in enumerate(trees[:64])])
    assert np.abs(zw[:64, 1] - host).max() <= 1e-12


def test_large_zones(gpu_lib):
    """The config-3 zone (shared memory, one step per CTA), a zone of the second class and one above the
    shared-memory size (global scratch), next to a small zone."""
    T = 96
    zones = [radial_feeder(n, seed=n, r_scale=0.07) for n in (10000, 15000, 25000)] + [synthetic_feeder(40, seed=1)]
    assert [z.n_nodes for z in zones[:3]] == [14100, 21150, 35250]
    rng = np.random.default_rng(0)
    P = rng.uniform(0.0, 3.0, (sum(z.n_res for z in zones), T))
    with _solver(gpu_lib, zones, T) as s:
        got = s.network_check(P, vset=1.03, full=True, zones=True)
    off = np.concatenate([[0], np.cumsum([z.n_res for z in zones])])
    for (a, b), z, h0, h1 in zip(_blocks(zones), zones, off[:-1], off[1:]):
        F, D = NR.zone_state(z.parent, z.r, z.res_node, P[h0:h1])
        assert np.array_equal(got["voltage"][a:b], np.sqrt(1.03 * 1.03 - D))
        assert np.abs(got["loading"][a:b] - F).max() <= 1e-12 * np.abs(F).max()
        drop = z.drop(P[h0:h1])
        v_res = np.sqrt(1.03 * 1.03 - drop)
        assert np.abs(got["voltage"][a:b][z.res_node] - v_res).max() <= 1e-12 * np.abs(drop).max()


@pytest.mark.parametrize("host", [False, True])
def test_pipelines_equal_one_solver(gpu_lib, host):
    trees, hm, cost, T = _refshape(6)
    N = sum(t.n_nodes for t in trees)
    scale = np.random.default_rng(1).uniform(-0.02, 0.02, N)
    kw = dict(vset=1.03, vlow=0.95, vhigh=1.05, scale=scale, full=True, zones=True)
    with _solved(gpu_lib, trees, hm, cost, T, **BENCH) as a:
        src = a.results()["P_sch"] * 1.5 if host else "schedule"
        ra = a.network_check(src, **kw)
    with _solved(gpu_lib, trees, hm, cost, T, cls=lambda sizes, T: gpu_lib.PipelinedSolver(sizes, T, pipelines=4),
                 **BENCH) as b:
        assert len(b.parts) == 4
        rb = b.network_check(src, **kw)
    assert ra["summary"] == rb["summary"]
    for k in ("voltage", "loading", "zone_worst"):
        assert np.array_equal(ra[k], rb[k]), k


def test_deterministic_and_without_side_effects(gpu_lib):
    trees, hm, cost, T = _refshape(2)
    with _solved(gpu_lib, trees, hm, cost, T, **BENCH) as s:
        before, est = s.results(), s.estimate()
        n0 = s.stats()["kernel_launches"]
        a = s.network_check("schedule", vset=1.03, full=True, zones=True)
        assert s.stats()["kernel_launches"] > n0
        b = s.network_check("schedule", vset=1.03, full=True, zones=True)
        assert ctypes_bytes(a) == ctypes_bytes(b)
        after, est2 = s.results(), s.estimate()
        for k in before:
            assert np.array_equal(before[k], after[k]), k
        assert all(np.array_equal(x, y) for x, y in zip(est, est2))
        s.solve_admm(**BENCH)
        again = s.results()
        for k in before:
            assert np.array_equal(before[k], again[k]), k


def ctypes_bytes(r):
    return (repr(sorted(r["summary"].items())), r["voltage"].tobytes(), r["loading"].tobytes(), r["zone_worst"].tobytes())


def test_argument_errors(gpu_lib):
    T = 24
    zones = _mixed_zones(1)[:2]
    hm = synthetic_homes(sum(z.n_res for z in zones), T, seed=2)

    def code(fn):
        with pytest.raises(gpu_lib.RevsError) as e:
            fn()
        assert e.value.code == 1, str(e.value)
        return str(e.value)

    with gpu_lib.Solver([z.n_res for z in zones], T) as s:
        s.set_feeder_tree(0, zones[0].parent, zones[0].r, zones[0].res_node)
        s.set_sensitivity(1, np.eye(zones[1].n_res) * 1e-3)
        assert "zone 1" in code(lambda: s.network_check(np.zeros((s.H, T))))
    with _solver(gpu_lib, zones, T) as s:
        s.set_homes(**hm)
        s.set_tariff(synthetic_tariff(T))
        code(lambda: s.network_check("schedule"))
        code(lambda: s.network_check("estimate"))
        P = np.zeros((s.H, T))
        code(lambda: s.network_check(P, vset=1.0, vlow=1.01, vhigh=1.05))
        code(lambda: s.network_check(P, vset=1.05, vlow=0.95, vhigh=1.05))
        summ = gpu_lib.NetworkSummary()
        for src, p in ((gpu_lib.REVS_NET_HOST, None), (7, P.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))):
            rc = s.lib.revs_network_check(s._h, src, p, 1.0, 0.95, 1.05, 1e-9, None, None, None, None, ctypes.byref(summ))
            assert rc == 1
        s.network_check(P)                                   # the solver still works

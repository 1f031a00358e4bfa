"""Host-side logic and the C-ABI surface, no GPU needed."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import INPUT, ROOT


def test_cabi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "revs_admm.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(revs_[a-z_0-9]+)\s*\(", hdr))
    assert len(declared) >= 20
    lib_path = os.path.join(ROOT, "revs-admm_b200", "librevs_admm.so")
    if not os.path.exists(lib_path):
        import __graft_entry__ as g
        g.build()
    lib = ctypes.CDLL(lib_path)
    for name in declared:
        assert hasattr(lib, name), name
    from revs_admm_b200 import _cabi
    assert declared == set(_cabi.SIGNATURES)


def test_no_cpu_fallback_without_gpu():
    import revs_admm_b200 as r
    try:
        n = r.device_count()
    except r.RevsError:
        n = 0
    if n > 0:
        pytest.skip("a GPU is visible")
    with pytest.raises(r.RevsError):
        r.Solver([4], 24)
    with pytest.raises(r.RevsError):
        r.contract(np.eye(4), np.eye(4))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "revs-admm_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "revs_oracle" not in txt.replace("oracle/revs_oracle.py", ""), f


def test_extract_formats(tmp_path):
    from revs_admm_b200 import extract
    tariff = extract.GetTariff(INPUT, "DVP", 6)
    assert len(tariff) == 24 and tariff[0] == 0.095111 and tariff[9] == 0.214357
    com = extract.GetCommunity(f"{INPUT}/121144-com.txt", 2)
    assert len(com) == 297
    homes = extract.GetHomeLoad(INPUT, 121, 6)
    assert len(homes) == 1126 and all(len(v) == 24 for v in homes.values())
    g = extract.GetDistNet(INPUT, 121144)
    assert g.number_of_nodes() == 1692 and g.number_of_edges() == 1691
    with pytest.raises(ValueError):
        extract.GetTariff(INPUT, "nope", 6)
    hp = extract.get_homes_ev_param(homes, g, com[:3], 4.8, 20, 0.2, 11, 23)
    assert hp[com[0]]["EV"] == dict(rating=4.8, capacity=20.0, initial=0.2, start=11, end=23)
    assert sum(bool(v["EV"]) for v in hp.values()) == 3
    # result file round trip
    P = {h: np.arange(24.0) + h % 7 for h in com[:5]}
    E = {h: np.zeros(24) for h in com[:3]}
    S = {h: np.linspace(0.2, 0.92, 25) for h in com[:3]}
    diff = {1: {h: 0.5 for h in com[:3]}, 2: {h: 0.25 for h in com[:3]}}
    path = tmp_path / "r.txt"
    path.write_text(extract.combine_result(P, E, S, com[:3], diff))
    back = extract.read_result(str(path))
    assert list(back) == ["Residence Usage Profile", "EV Charger Usage Profile",
                          "EV Charger State of Charge Profile", "EV Convergence over Iterations"]
    assert np.array_equal(back["Residence Usage Profile"][com[4]], P[com[4]])
    assert np.array_equal(back["EV Convergence over Iterations"][com[0]], [0.5, 0.25])


def test_tree_from_graph_and_synthetic():
    from revs_admm_b200 import extract
    from revs_admm_b200.feeder import synthetic_feeder, synthetic_homes, synthetic_tariff, tree_from_graph
    g = extract.GetDistNet(INPUT, 121144)
    t = tree_from_graph(g)
    assert t.n_nodes == 1691 and t.n_res == 1126
    assert (t.parent < np.arange(t.n_nodes)).all() and (t.parent >= -1).all()
    assert (t.parent == -1).sum() == 5            # five feeder lines leave the substation
    s = synthetic_feeder(1000, seed=3)
    assert s.n_res == 1000 and (s.parent < np.arange(s.n_nodes)).all()
    hm = synthetic_homes(1000, 96, seed=3)
    assert hm["load"].shape == (1000, 96) and hm["load"].min() > 0
    assert 0.85 < hm["has_ev"].mean() < 0.95
    assert len(synthetic_tariff(96)) == 96 and len(synthetic_tariff(24)) == 24


def test_revs_fixture_interface(case121144):
    fx = case121144["fx"]
    assert fx.com == 2 and fx.optim == "distributed"
    assert fx.out_dir.endswith("121144-com2/distributed")
    assert len(case121144["saved"]["ev_homes"]) == 267
    with pytest.raises(NotImplementedError):
        fx.plot_result({}, case121144["dist"])            # plotting is out of scope
    # no CPU fallback: without a GPU the centralized entry point fails loudly in the library, not silently on the host
    from revs_admm_b200 import RevsError, device_count
    try:
        n_gpu = device_count()
    except RevsError:
        n_gpu = 0
    if n_gpu == 0:
        with pytest.raises(RevsError):
            fx.get_centralized_optimal(case121144["tariff"], case121144["homes"], case121144["dist"])


def test_config_yaml_has_the_reference_schema():
    """revs_config.yaml: the key set of the reference's file (revs_config.yaml:1-39), including the
    draw_parameters / init_parameters blocks its test-optimizer.py:25 reads."""
    import os
    import yaml
    from conftest import ROOT
    cfg = yaml.safe_load(open(os.path.join(ROOT, "revs-admm_b200", "revs_config.yaml")))
    assert set(cfg) == {"run_parameters", "init_parameters"}
    run = cfg["run_parameters"]
    assert set(run) == {"input_filepath", "input_parameters", "optimizer_parameters", "draw_parameters"}
    assert set(run["input_filepath"]) == {"data_path", "out_path", "fig_path", "grb_path", "regionID", "networkID",
                                          "communityID", "tariffID", "optimizer_mode"}
    assert set(run["input_parameters"]) == {"adoption", "rating", "seed", "capacity", "initial_soc", "start_time",
                                            "end_time", "shift_time"}
    assert set(run["optimizer_parameters"]) == {"v0", "vmin", "vmax", "max_iterations", "kappa"}
    assert set(run["draw_parameters"]) == {"figwidth", "figheight", "fontsize", "labelsize", "tick_labelsize"}
    assert set(cfg["init_parameters"]) == {"nodes", "module"}


def test_pipeline_cuts_cover_all_zones():
    """parallel.PipelinedSolver cuts the zone list with shard_feeders: contiguous, complete, home-balanced."""
    from revs_admm_b200.parallel import shard_feeders
    rng = np.random.default_rng(0)
    sizes = rng.integers(40, 170, size=1250)
    for K in (1, 2, 3, 4, 8):
        cuts = [shard_feeders(sizes, K, k) for k in range(K)]
        assert cuts[0][0] == 0 and cuts[-1][1] == len(sizes)
        assert all(cuts[k][1] == cuts[k + 1][0] for k in range(K - 1))
        homes = [int(sizes[a:b].sum()) for a, b in cuts]
        assert max(homes) - min(homes) <= 2 * sizes.max()


def test_objective_sandwich_lower_bound():
    """bench.objective_check: the cost of the cheapest SOC-feasible schedule without voltage limits is a
    lower bound of any feasible schedule's cost; the load-only schedule (no charging) is below it."""
    import bench
    trees, hm, cost, sizes, T = bench.make_rank_problem("tiny", 0)
    dist, lb, viol = bench.objective_check(trees, hm, cost, hm["load"].copy(), T)
    assert dist < lb                                   # no charging at all is cheaper than any feasible schedule
    # a feasible schedule: every EV home charges in its n_min cheapest window hours -> cost == lower bound
    P = hm["load"].copy()
    step = hm["rating"] / np.maximum(hm["capacity"], 1e-300)
    for h in np.nonzero(hm["has_ev"])[0]:
        nmin = max(int(np.ceil((0.9 - hm["initial"][h]) / step[h] - 1e-9)), 0)
        win = np.arange(hm["start"][h], hm["end"][h])
        pick = win[np.argsort(np.asarray(cost)[win], kind="stable")[:nmin]]
        P[h, pick] += hm["rating"][h]
    dist2, lb2, _ = bench.objective_check(trees, hm, cost, P, T)
    assert lb2 == lb and abs(dist2 - lb) <= 1e-9 * abs(lb)


@pytest.mark.parametrize("H", [300, 20000])
def test_dump_outputs_writes_a_fixed_sample(tmp_path, H):
    """bench --dump-outputs: every result array of the solver as float64 .npy, rows (diff: columns) of the same
    seeded sample of homes in every run, the whole population when it is small."""
    import bench
    T, iters = 96, 15
    rng = np.random.default_rng(2)
    res = dict(P_sch=rng.random((H, T)), P_ev=rng.random((H, T)), SOC=rng.random((H, T + 1)), diff=rng.random((iters, H)))
    est = rng.random((H, T)), rng.random((H, T))

    class Fake:
        def results(self): return dict(res)
        def estimate(self): return est
    fake = Fake()
    fake.H = H
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), fake)
    n = min(H, bench.DUMP_HOMES)
    idx = np.load(tmp_path / "a" / "home_index.npy")
    assert idx.dtype == np.float64 and len(np.unique(idx)) == n
    rows = idx.astype(np.int64)
    want = dict(res, P_est=est[0], Gamma=est[1])
    for name, a in want.items():
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert got.dtype == np.float64
        assert np.array_equal(got, a[:, rows] if name == "diff" else a[rows]), name
        assert np.array_equal(got, np.load(tmp_path / "b" / f"{name}.npy")), name
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 << 20


def test_pipelined_stats_combination():
    """PipelinedSolver.stats(): counters add up, total_ms is the longest pipeline, residuals recombine as RMS."""
    from revs_admm_b200.parallel import PipelinedSolver

    class Fake:
        def __init__(self, d): self.d = d
        def stats(self): return dict(self.d)

    ps = PipelinedSolver.__new__(PipelinedSolver)
    ps.parts = [Fake(dict(kernel_launches=10, total_ms=3.0, admm_iterations=5, max_working_set=4, primal_residual=1.0, dual_residual=2.0, qp_ms=1.5)),
                Fake(dict(kernel_launches=7, total_ms=4.0, admm_iterations=5, max_working_set=9, primal_residual=3.0, dual_residual=0.0, qp_ms=0.5))]
    ps.rows = [(0, 100), (100, 400)]
    st = ps.stats()
    assert st["kernel_launches"] == 17 and st["total_ms"] == 4.0 and st["total_ms_sum"] == 7.0 and st["max_working_set"] == 9
    assert st["pipelines"] == 2 and st["qp_ms"] == 2.0
    assert abs(st["primal_residual"] - np.sqrt((1.0 * 100 + 9.0 * 300) / 400)) < 1e-12
    ps.parts = []          # nothing to close
    ps.pool = None


def test_pack_trees_concatenates_the_zone_arrays():
    """Solver.pack_trees (the interpreter-side half of revs_set_feeder_trees, done pipeline by pipeline in
    PipelinedSolver.schedule): node offsets, parents, resistances and residence nodes of all zones back to back, in the
    dtypes the C ABI takes."""
    from revs_admm_b200._cabi import Solver
    from revs_admm_b200.feeder import synthetic_feeder
    trees = [synthetic_feeder(n, seed=i, r_secondary=1e-3) for i, n in enumerate([20, 7, 33])]
    s = Solver.__new__(Solver)                       # no device: only the packing is exercised
    s.nf, s.H = 3, 60
    off, parent, r, res = s.pack_trees(trees)
    assert off.dtype == np.int64 and parent.dtype == np.int32 and r.dtype == np.float64 and res.dtype == np.int32
    assert off.tolist() == [0] + list(np.cumsum([len(t.parent) for t in trees]))
    for i, t in enumerate(trees):
        assert np.array_equal(parent[off[i]:off[i + 1]], t.parent) and np.array_equal(r[off[i]:off[i + 1]], t.r)
    assert len(res) == 60 and np.array_equal(res[20:27], trees[1].res_node)
    s._h = None                                      # nothing to destroy

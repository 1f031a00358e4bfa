"""GPU edge cases: ragged shapes, degenerate populations, option/exactness cross-checks, errors."""
import numpy as np
import pytest

import revs_oracle as O

pytestmark = pytest.mark.gpu


def _problem(sizes, T, seed, r_secondary=1e-3, **hkw):
    from revs_admm_b200.feeder import synthetic_feeder, synthetic_homes, synthetic_tariff
    trees = [synthetic_feeder(n, seed=seed + i, r_secondary=r_secondary, laterals=max(1, min(5, n))) for i, n in enumerate(sizes)]
    hm = synthetic_homes(sum(sizes), T, seed=seed, **hkw)
    return trees, hm, synthetic_tariff(T) if T >= 24 else np.linspace(0.05, 0.2, T)


def _oracle(trees, hm, cost, kw):
    Rb = [O.rmat_from_tree(t.parent, t.r)[np.ix_(t.res_node, t.res_node)] for t in trees]
    return O.solve_ADMM_arrays(Rb, load=hm["load"], cost=cost, ev_mask=hm["has_ev"].astype(bool), rating=hm["rating"],
                               capacity=hm["capacity"], initial=hm["initial"], start=hm["start"], end=hm["end"], **kw)


def _gpu(lib, sizes, T, trees, hm, cost, kw, screen=1, newton_min_n=None):
    with lib.Solver(sizes, T) as s:
        s.set_option("screen", screen)
        if newton_min_n is not None:
            s.set_option("newton_min_n", newton_min_n)
        s.set_feeder_trees(trees)
        s.set_homes(**hm)
        s.set_tariff(cost)
        done = s.solve_admm(**kw)
        out = s.results(done)
        out["P_est"], out["Gamma"] = s.estimate()
        out["stats"] = s.stats()
    return out


@pytest.mark.parametrize("sizes,T", [([1], 24), ([17, 1, 33], 24), ([5, 3], 7), ([40], 1), ([30, 21], 100), ([12], 256)])
def test_ragged_shapes_match_oracle(gpu_lib, sizes, T):
    trees, hm, cost = _problem(sizes, T, seed=sum(sizes) + T)
    if T < 24:      # plug-in window must fit the horizon
        hm["start"][:] = 0
        hm["end"][:] = T
        hm["capacity"][:] = 4.8 * max(1, T // 2) / 0.75      # ~T/2 charging steps needed
    kw = dict(kappa=5.0, iter_max=4, vset=1.0, vlow=0.95, vhigh=1.02)
    out = _gpu(gpu_lib, sizes, T, trees, hm, cost, kw)
    ref = _oracle(trees, hm, cost, kw)
    assert np.array_equal(out["P_ev"], ref["P_ev"])
    assert np.abs(out["P_sch"] - ref["P_sch"]).max() <= 1e-4
    assert np.abs(out["P_est"] - ref["P_est"]).max() <= 1e-4
    assert np.abs(out["diff"] - ref["diff"]).max() <= 1e-7
    assert np.allclose(out["SOC"], ref["SOC"], atol=1e-12)


@pytest.mark.parametrize("adoption", [0.0, 1.0])
def test_no_ev_and_all_ev(gpu_lib, adoption):
    sizes, T = [60, 45], 24
    trees, hm, cost = _problem(sizes, T, seed=9, adoption=adoption)
    kw = dict(kappa=5.0, iter_max=5, vset=1.0, vlow=0.95, vhigh=1.02)
    out = _gpu(gpu_lib, sizes, T, trees, hm, cost, kw)
    ref = _oracle(trees, hm, cost, kw)
    assert np.array_equal(out["P_ev"], ref["P_ev"])
    assert np.abs(out["P_sch"] - ref["P_sch"]).max() <= 1e-4
    if adoption == 0.0:
        assert np.array_equal(out["P_sch"], hm["load"]) and out["SOC"].max() == 0.0


def test_screening_is_exact(gpu_lib):
    """BF16 screening + FP64 recheck must give bit-identical results to the FP64 contraction."""
    sizes, T = [130, 77, 201], 96
    trees, hm, cost = _problem(sizes, T, seed=21)
    kw = dict(kappa=5.0, iter_max=6, vset=1.0, vlow=0.95, vhigh=1.015)
    a = _gpu(gpu_lib, sizes, T, trees, hm, cost, kw, screen=1)
    b = _gpu(gpu_lib, sizes, T, trees, hm, cost, kw, screen=0)
    for k in ("P_sch", "P_ev", "SOC", "diff", "P_est", "Gamma"):
        assert np.array_equal(a[k], b[k]), k
    assert a["stats"]["gemm_launches"] == b["stats"]["gemm_launches"] > 0


def test_dense_block_input_equals_tree_input(gpu_lib):
    sizes, T = [48, 31], 24
    trees, hm, cost = _problem(sizes, T, seed=5)
    kw = dict(kappa=5.0, iter_max=4, vset=1.0, vlow=0.95, vhigh=1.02)
    a = _gpu(gpu_lib, sizes, T, trees, hm, cost, kw)
    with gpu_lib.Solver(sizes, T) as s:
        for f, t in enumerate(trees):
            s.set_sensitivity(f, O.rmat_from_tree(t.parent, t.r)[np.ix_(t.res_node, t.res_node)])
        s.set_homes(**hm)
        s.set_tariff(cost)
        done = s.solve_admm(**kw)
        b = s.results(done)
    assert np.array_equal(a["P_ev"], b["P_ev"])
    assert np.abs(a["P_sch"] - b["P_sch"]).max() <= 1e-9


def test_reliability_kinds_on_synthetic_tree(gpu_lib):
    from revs_admm_b200.feeder import synthetic_feeder
    T = 24
    t = synthetic_feeder(75, seed=3, r_secondary=1e-3)
    rng = np.random.default_rng(0)
    P = rng.uniform(0, 6, (75, T))
    R = O.rmat_from_tree(t.parent, t.r)
    Pall = np.zeros((t.n_nodes, T))
    Pall[t.res_node] = P
    with gpu_lib.Solver([75], T) as s:
        s.set_feeder_tree(0, t.parent, t.r, t.res_node)
        rows = np.arange(t.n_nodes)
        drop = s.reliability(0, 2, rows, P=P)
        volt = s.reliability(0, 0, rows, vset=1.03, P=P)
        flow = s.reliability(0, 1, rows, P=P, scale=np.full(t.n_nodes, 0.5))
        with pytest.raises(gpu_lib.RevsError):
            s.reliability(0, 0, [t.n_nodes], P=P)
    assert np.abs(drop - R @ Pall).max() <= 1e-12
    assert np.abs(volt - np.sqrt(1.03 ** 2 - R @ Pall)).max() <= 1e-12
    # flow on the edge above node i = load of its subtree
    sub = Pall.copy()
    for i in range(t.n_nodes - 1, -1, -1):
        if t.parent[i] >= 0:
            sub[t.parent[i]] += sub[i]
    assert np.abs(flow - 0.5 * sub).max() <= 1e-10


def test_argument_errors(gpu_lib):
    from revs_admm_b200.feeder import synthetic_feeder, synthetic_homes
    with pytest.raises(gpu_lib.RevsError):
        gpu_lib.Solver([4], 300)                       # horizon limit
    with gpu_lib.Solver([20], 24) as s:
        with pytest.raises(gpu_lib.RevsError):         # nothing set yet
            s.solve_admm()
        t = synthetic_feeder(20, seed=1)
        s.set_feeder_tree(0, t.parent, t.r, t.res_node)
        s.set_homes(**synthetic_homes(20, 24, seed=1))
        s.set_tariff(np.ones(24))
        with pytest.raises(gpu_lib.RevsError):         # vhigh <= vset
            s.solve_admm(vset=1.05, vhigh=1.05)
        with pytest.raises(gpu_lib.RevsError):
            s.set_option("nonsense", 1)
        with pytest.raises(gpu_lib.RevsError):         # parent after child
            s.set_feeder_tree(0, t.parent[::-1].copy(), t.r, t.res_node)
        assert s.solve_admm(iter_max=2) == 2


def test_working_set_overflow_is_loud(gpu_lib):
    """More than 128 simultaneously binding voltage rows in one (feeder,hour) column is outside what the DENSE QP kernels
    hold in shared memory: forced onto them (newton_min_n above the zone size) the solve fails with REVS_ERR_NOCONV.
    By default a zone of this size given as a tree runs on the tree-Newton path, which has no such limit
    (test_gpu_newton.py::test_former_overflow_case_matches_oracle)."""
    from revs_admm_b200.feeder import synthetic_feeder, synthetic_homes, synthetic_tariff
    n, T = 1000, 24      # the oracle finds up to 149 binding rows per hour on this feeder
    t = synthetic_feeder(n, seed=0, laterals=5)
    hm = synthetic_homes(n, T, seed=77)
    with gpu_lib.Solver([n], T) as s:
        s.set_option("newton_min_n", 4096)
        s.set_feeder_tree(0, t.parent, t.r, t.res_node)
        s.set_homes(**hm)
        s.set_tariff(synthetic_tariff(T))
        with pytest.raises(gpu_lib.RevsError) as e:
            s.solve_admm(iter_max=4, vset=1.03, vlow=0.95, vhigh=1.05)
        assert e.value.code == 4


@pytest.mark.parametrize("sizes,vhigh", [([100, 200], 1.02), ([300], 1.02), ([297, 157, 257, 320, 129], 1.02), ([400], 1.02), ([600, 90], 1.05)])
def test_zone_size_classes_match_oracle(gpu_lib, sizes, vhigh):
    """Zones <= 128 / <= 256 / <= 320 (warp-per-column kernels, NJ = 4 / 6 / 8 / 10 -- the reference feeder's zones
    are 157..297), <= 512 (CTA kernel with in-kernel verification) and larger (CTA kernel + re-screening rounds)
    under limits tight enough to bind."""
    T = 24
    trees, hm, cost = _problem(sizes, T, seed=sum(sizes), r_secondary=1e-3)
    kw = dict(kappa=5.0, iter_max=5, vset=1.0, vlow=0.95, vhigh=vhigh)
    out = _gpu(gpu_lib, sizes, T, trees, hm, cost, kw, newton_min_n=4096)       # dense kernels for every size (tree-Newton: test_gpu_newton.py)
    ref = _oracle(trees, hm, cost, kw)
    assert out["stats"]["max_working_set"] >= 10         # the limits do bind (tens of rows per column)
    assert np.array_equal(out["P_ev"], ref["P_ev"])
    assert np.abs(out["P_sch"] - ref["P_sch"]).max() <= 1e-4
    assert np.abs(out["P_est"] - ref["P_est"]).max() <= 1e-4
    assert np.abs(out["diff"] - ref["diff"]).max() <= 1e-7


def test_many_binding_rows_hand_over(gpu_lib):
    """Working sets that outgrow the warp kernel (16 rows) and the first CTA class (32 rows):
    columns are handed from class to class and still land on the oracle's projection."""
    sizes, T = [120, 96], 12
    trees, hm, cost = _problem(sizes, T, seed=77, r_secondary=2e-3, adoption=1.0)
    hm["start"][:] = 0
    hm["end"][:] = T
    kw = dict(kappa=5.0, iter_max=4, vset=1.0, vlow=0.95, vhigh=1.02)
    out = _gpu(gpu_lib, sizes, T, trees, hm, cost, kw)
    ref = _oracle(trees, hm, cost, kw)
    assert out["stats"]["max_working_set"] > 16
    assert np.array_equal(out["P_ev"], ref["P_ev"])
    assert np.abs(out["P_est"] - ref["P_est"]).max() <= 1e-4
    assert np.abs(out["P_sch"] - ref["P_sch"]).max() <= 1e-4


def test_scheduling_options_do_not_change_results(gpu_lib):
    """Home solve in line vs on its own stream, solve_admm (iterations enqueued back to back) vs
    admm_begin/admm_step (host sync per iteration): bit-identical outputs."""
    sizes, T = [140, 60, 33], 48
    trees, hm, cost = _problem(sizes, T, seed=3)
    kw = dict(kappa=5.0, iter_max=6, vset=1.0, vlow=0.95, vhigh=1.015)
    base = _gpu(gpu_lib, sizes, T, trees, hm, cost, kw)
    with gpu_lib.Solver(sizes, T) as s:
        s.set_option("overlap_home", 0)
        s.set_feeder_trees(trees)
        s.set_homes(**hm)
        s.set_tariff(cost)
        s.admm_begin(**kw)
        for _ in range(kw["iter_max"]):
            s.admm_step()
        out = s.results(kw["iter_max"])
        out["P_est"], out["Gamma"] = s.estimate()
    for k in ("P_sch", "P_ev", "SOC", "diff", "P_est", "Gamma"):
        assert np.array_equal(base[k], out[k]), k


@pytest.mark.parametrize("pipelines", [2, 3, 7])
def test_pipelined_solver_equals_single_solver(gpu_lib, pipelines):
    """K stream pipelines over contiguous groups of zones (parallel.PipelinedSolver) return the single
    solver's results bit for bit: zones never exchange data."""
    sizes, T = [60, 45, 33, 80, 20], 24
    trees, hm, cost = _problem(sizes, T, seed=11)
    kw = dict(kappa=5.0, iter_max=5, vset=1.0, vlow=0.95, vhigh=1.015)
    base = _gpu(gpu_lib, sizes, T, trees, hm, cost, kw)
    with gpu_lib.PipelinedSolver(sizes, T, pipelines=pipelines) as s:
        s.set_feeder_trees(trees)
        s.set_homes(**hm)
        s.set_tariff(cost)
        done = s.solve_admm(**kw)
        out = s.results(done)
        out["P_est"], out["Gamma"] = s.estimate()
        st = s.stats()
    assert 2 <= st["pipelines"] <= min(pipelines, len(sizes)) and st["admm_iterations"] == kw["iter_max"]
    for k in ("P_sch", "P_ev", "SOC", "diff", "P_est", "Gamma"):
        assert np.array_equal(base[k], out[k]), k


@pytest.mark.parametrize("sizes,T,vhigh", [([140, 60, 33], 48, 1.015), ([300, 210], 24, 1.02), ([600, 90], 24, 1.05), ([120, 96], 12, 1.02)])
def test_captured_loop_equals_host_driven_loop(gpu_lib, sizes, T, vhigh):
    """revs_solve_admm from ONE captured graph (ADMM iterations and working-set rounds decided on the
    device, CTA classes behind IF nodes) against the host-driven loop (one host sync per round):
    bit-identical results, same number of working-set rounds -- including zones that need several rounds
    (> 512 residences: re-screening) and columns handed from class to class."""
    trees, hm, cost = _problem(sizes, T, seed=5 + sum(sizes), r_secondary=2e-3 if T == 12 else 1e-3,
                               **(dict(adoption=1.0) if T == 12 else {}))
    if T == 12:                                      # every charger may run in any step: working sets beyond the warp kernel
        hm["start"][:] = 0
        hm["end"][:] = T
    kw = dict(kappa=5.0, iter_max=6, vset=1.0, vlow=0.95, vhigh=vhigh)
    outs, rounds = [], []
    for graph in (1, 0):
        with gpu_lib.Solver(sizes, T) as s:
            s.set_option("graph", graph)
            s.set_option("newton_min_n", 4096)            # zones above 512 on the dense kernels (tree-Newton: test_gpu_newton.py)
            s.set_feeder_trees(trees)
            s.set_homes(**hm)
            s.set_tariff(cost)
            for rep in range(2):                      # the second run re-launches the instantiated graph
                done = s.solve_admm(**kw)
            out = s.results(done)
            out["P_est"], out["Gamma"] = s.estimate()
            st = s.stats()
            assert done == kw["iter_max"] and st["admm_iterations"] == done and st["kernel_launches"] > 5 * done
            rounds.append(st["qp_outer_iterations"])
            outs.append(out)
    for k in ("P_sch", "P_ev", "SOC", "diff", "P_est", "Gamma"):
        assert np.array_equal(outs[0][k], outs[1][k]), k
    assert rounds[0] == rounds[1]
    assert rounds[0] >= kw["iter_max"]               # the dense kernels run at least one working-set round per iteration


@pytest.mark.parametrize("sizes,T", [([70, 45, 33], 96), ([40, 21], 24), ([30], 100), ([12], 256)])
def test_residual_sums_follow_the_iterates(gpu_lib, sizes, T):
    """The residual sums of the stopping rule (lpsolver.py:280-284 restated as ADMM residuals): primal = sum (P_est[k+1] -
    P_sch[k+1])^2, dual = sum (P_sch[k+1] - P_sch[k])^2 with P_sch[0] = 0.  The dual sum is accumulated per home by
    home_solve_kernel and only added up by dual_update_kernel: checked against the downloaded schedules after every
    iteration, and the captured loop must end on the same values as the stepped one."""
    trees, hm, cost = _problem(sizes, T, seed=3 + sum(sizes))
    kw = dict(kappa=5.0, iter_max=5, vset=1.0, vlow=0.95, vhigh=1.02)
    H = sum(sizes)
    with gpu_lib.Solver(sizes, T) as s:
        s.set_feeder_trees(trees)
        s.set_homes(**hm)
        s.set_tariff(cost)
        s.admm_begin(**kw)
        prev = np.zeros((H, T))
        for k in range(kw["iter_max"]):
            sums = s.admm_step()
            P = s.results(k + 1)["P_sch"]
            P_est, _ = s.estimate()
            want_d, want_p = ((P - prev) ** 2).sum(), ((P_est - P) ** 2).sum()
            assert abs(sums[1] - want_d) <= 1e-12 * max(1.0, want_d), (k, sums[1], want_d)
            assert abs(sums[0] - want_p) <= 1e-12 * max(1.0, want_p), (k, sums[0], want_p)
            assert sums[2] == H * T
            prev = P
        st_step = s.stats()
        s.solve_admm(**kw)                              # captured loop
        st_loop = s.stats()
    assert st_loop["dual_residual"] == st_step["dual_residual"] and st_loop["primal_residual"] == st_step["primal_residual"]
    assert abs(st_step["dual_residual"] - kw["kappa"] * np.sqrt(want_d / (H * T))) <= 1e-12 * max(1.0, st_step["dual_residual"])


def test_captured_loop_stops_on_the_device(gpu_lib):
    """tol > 0: the last CTA of dual_update_kernel clears the loop condition; same iteration count and
    results as the host-driven loop, and an infeasible home stops the loop with REVS_ERR_INFEASIBLE."""
    from revs_admm_b200.feeder import synthetic_feeder, synthetic_homes, synthetic_tariff
    n, T = 50, 24
    t = synthetic_feeder(n, seed=2, r_secondary=1e-5)
    hm = synthetic_homes(n, T, seed=2)
    res = []
    for graph in (1, 0):
        with gpu_lib.Solver([n], T) as s:
            s.set_option("graph", graph)
            s.set_feeder_tree(0, t.parent, t.r, t.res_node)
            s.set_homes(**hm)
            s.set_tariff(synthetic_tariff(T))
            done = s.solve_admm(iter_max=40, tol=1e-6)
            st = s.stats()
            assert 1 < done < 40 and st["primal_residual"] < 1e-6 and st["dual_residual"] < 1e-6
            res.append((done, s.results(done)))
    assert res[0][0] == res[1][0]
    for k in ("P_sch", "P_ev", "diff"):
        assert np.array_equal(res[0][1][k], res[1][1][k])
    hm["end"][:] = hm["start"] + 1                   # one-step window: SOC target unreachable
    with gpu_lib.Solver([n], T) as s:
        s.set_feeder_tree(0, t.parent, t.r, t.res_node)
        s.set_homes(**hm)
        s.set_tariff(synthetic_tariff(T))
        with pytest.raises(gpu_lib.RevsError) as e:
            s.solve_admm(iter_max=5)
        assert e.value.code == 3


def test_pipelined_solver_global_stopping_rule(gpu_lib):
    """tol > 0 with several pipelines: lock-step iterations, residual sums combined between steps --
    the iteration count and every result equal the single solver's (ADVICE r1: pipelines used to stop
    on their own residuals)."""
    from revs_admm_b200.feeder import synthetic_feeder, synthetic_homes, synthetic_tariff
    sizes, T = [50, 40, 30, 60], 24
    trees = [synthetic_feeder(n, seed=20 + i, r_secondary=(1e-5 if i % 2 else 4e-5)) for i, n in enumerate(sizes)]
    hm = synthetic_homes(sum(sizes), T, seed=21)
    cost = synthetic_tariff(T)
    kw = dict(kappa=5.0, iter_max=60, vset=1.0, vlow=0.95, vhigh=1.05, tol=1e-5)
    with gpu_lib.Solver(sizes, T) as s:
        s.set_feeder_trees(trees)
        s.set_homes(**hm)
        s.set_tariff(cost)
        done1 = s.solve_admm(**kw)
        one = s.results(done1)
    with gpu_lib.PipelinedSolver(sizes, T, pipelines=3) as s:
        s.set_feeder_trees(trees)
        s.set_homes(**hm)
        s.set_tariff(cost)
        done3 = s.solve_admm(**kw)
        three = s.results()
        with pytest.raises(ValueError):
            s.results(out=dict(P_sch=np.empty((sum(sizes), T)), P_ev=np.empty((sum(sizes), T)),
                               SOC=np.empty((sum(sizes), T + 1)), diff=np.empty((done3 - 1, sum(sizes)))))
    assert 1 < done1 < 60 and done3 == done1
    for k in ("P_sch", "P_ev", "SOC"):
        assert np.array_equal(one[k], three[k]), k
    assert np.array_equal(one["diff"][:done1], three["diff"][:done1])


def test_results_buffer_capacity_is_checked(gpu_lib):
    """revs_get_results refuses a diff buffer with fewer rows than iterations ran (ADVICE r1)."""
    sizes, T = [20], 24
    trees, hm, cost = _problem(sizes, T, seed=1)
    with gpu_lib.Solver(sizes, T) as s:
        s.set_feeder_trees(trees)
        s.set_homes(**hm)
        s.set_tariff(cost)
        s.solve_admm(iter_max=4)
        out = dict(P_sch=np.empty((20, T)), P_ev=np.empty((20, T)), SOC=np.empty((20, T + 1)), diff=np.empty((3, 20)))
        with pytest.raises(gpu_lib.RevsError) as e:
            s.results(out=out)
        assert e.value.code == 1
        with pytest.raises(ValueError):
            s.results(out=dict(out, P_sch=np.empty((20, T), dtype=np.float32)))


def test_compact_schedule_download_equals_full_results(gpu_lib):
    """revs_get_schedule (P_sch + charging bit masks + diff) and expand_schedule on the host give exactly
    the arrays of revs_get_results, for a single solver and through PipelinedSolver.schedule(compact=True)."""
    sizes, T = [70, 45, 33], 96
    trees, hm, cost = _problem(sizes, T, seed=9)
    kw = dict(kappa=5.0, iter_max=4, vset=1.0, vlow=0.95, vhigh=1.015)
    with gpu_lib.Solver(sizes, T) as s:
        s.set_feeder_trees(trees)
        s.set_homes(**hm)
        s.set_tariff(cost)
        done = s.solve_admm(**kw)
        full = s.results(done)
        comp = s.schedule_compact()
    assert comp["mask"].shape == (sum(sizes), 2) and comp["mask"].dtype == np.uint64
    p_ev, soc = gpu_lib.expand_schedule(comp["mask"], T, hm["has_ev"], hm["rating"], hm["capacity"], hm["initial"])
    assert np.array_equal(comp["P_sch"], full["P_sch"]) and np.array_equal(comp["diff"], full["diff"])
    assert np.array_equal(p_ev, full["P_ev"]) and np.array_equal(soc, full["SOC"])
    with gpu_lib.PipelinedSolver(sizes, T, pipelines=2) as ps:
        out = ps.schedule(trees, hm, cost, compact=True, **kw)
    assert np.array_equal(out["P_sch"], full["P_sch"]) and np.array_equal(out["mask"], comp["mask"])
    assert np.array_equal(out["diff"][:done], full["diff"])


@pytest.mark.parametrize("sizes,T,vhigh", [([140, 60, 33], 48, 1.015), ([297, 157, 257, 320, 129], 24, 1.02), ([120, 96], 12, 1.02), ([1, 2, 31, 33], 24, 1.01)])
def test_warp_zone_sizes_match_oracle(gpu_lib, sizes, T, vhigh):
    """The dense kernels (BF16 screening + FP64 rows of R) on zones on both sides of every size-class boundary of the
    warp kernels (128 / 129, 256 / 257, 320) against the oracle: identical charging hours, estimates within 1e-6 kW,
    binding working sets of two rows or more."""
    trees, hm, cost = _problem(sizes, T, seed=13 + sum(sizes), r_secondary=2e-3 if T == 12 else 1e-3,
                               **(dict(adoption=1.0) if T == 12 else {}))
    if T == 12:
        hm["start"][:] = 0
        hm["end"][:] = T
    kw = dict(kappa=5.0, iter_max=6, vset=1.0, vlow=0.95, vhigh=vhigh)
    out = _gpu(gpu_lib, sizes, T, trees, hm, cost, kw)
    ref = _oracle(trees, hm, cost, kw)
    assert np.array_equal(out["P_ev"], ref["P_ev"])
    assert np.abs(out["P_est"] - ref["P_est"]).max() <= 1e-6
    assert np.abs(out["diff"] - ref["diff"]).max() <= 1e-7
    assert out["stats"]["max_working_set"] >= 2


def test_sharded_reliability_on_one_rank_equals_plain_check(gpu_lib):
    """revs_reliability_sharded with a world of one (the gather buffer attached to itself): the contraction epilogue
    stores through the gather path, the result equals revs_reliability bit for bit.  (Two and more ranks:
    tests/mgpu_check.py on a multi-GPU box.)"""
    from revs_admm_b200.feeder import synthetic_feeder
    from revs_admm_b200.parallel import attach_gather
    T = 24
    t = synthetic_feeder(700, seed=12, r_secondary=2e-4)
    P = np.random.default_rng(1).random((700, T)) * 2.0
    rows = np.arange(t.n_nodes, dtype=np.int32)
    with gpu_lib.Solver([700], T) as s:
        s.set_feeder_tree(0, t.parent, t.r, t.res_node)
        with pytest.raises(gpu_lib.RevsError):
            s.reliability_sharded(0, gpu_lib.REVS_REL_DROP, rows, P)        # no gather buffer yet
        assert attach_gather(s, len(rows) * T) == 1
        for kind in (gpu_lib.REVS_REL_VOLTAGE, gpu_lib.REVS_REL_FLOW, gpu_lib.REVS_REL_DROP):
            a = s.reliability(0, kind, rows, vset=1.03, P=P)
            for _ in range(2):
                assert np.array_equal(s.reliability_sharded(0, kind, rows, P, vset=1.03), a)
        with pytest.raises(gpu_lib.RevsError):
            s.reliability_sharded(0, gpu_lib.REVS_REL_DROP, np.arange(t.n_nodes, dtype=np.int32).repeat(2), P)   # beyond the buffer

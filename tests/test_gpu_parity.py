"""GPU parity tests: the CUDA path through the C ABI against the CPU oracle.

Tolerances are the ones BASELINE.json's north_star states: schedules <= 1e-4 kW per
home-hour, voltages <= 1e-5 pu, objective rel. <= 1e-6; integer decisions (which hours a
charger is on) must be identical.
"""
import numpy as np
import pytest

import revs_oracle as O

pytestmark = pytest.mark.gpu

TOL_KW = 1e-4
TOL_PU = 1e-5


def _arrays(homes, res):
    from revs_admm_b200.lpsolver import _home_arrays
    return _home_arrays(homes, res)


def _oracle_kwargs(a):
    return dict(load=a["load"], ev_mask=a["has_ev"].astype(bool), rating=a["rating"],
                capacity=a["capacity"], initial=a["initial"], start=a["start"], end=a["end"])


# ----------------------------------------------------------------- contraction
@pytest.mark.parametrize("M,K,T", [(1, 1, 1), (7, 5, 3), (64, 16, 24), (130, 100, 24), (200, 333, 48),
                                   (129, 1000, 96), (1126, 1126, 24), (300, 257, 100)])
def test_contract_matches_numpy(gpu_lib, M, K, T):
    rng = np.random.default_rng(M * 1000 + K + T)
    A, B = rng.standard_normal((M, K)), rng.standard_normal((K, T))
    C = gpu_lib.contract(A, B)
    ref = A @ B
    assert np.abs(C - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max()) * np.sqrt(K)


# ----------------------------------------------------------------- home step
def test_home_step_bit_exact_random(gpu_lib):
    from revs_admm_b200.feeder import synthetic_homes, synthetic_tariff
    for T, H, slow in [(24, 257, False), (96, 130, False), (40, 33, False), (96, 77, True)]:
        hm = synthetic_homes(H, T, seed=T, rating_kw=1.2 if slow else 4.8)   # slow: 47..53 hours -> ranking path
        if T == 40:
            hm["start"][:] = 3
            hm["end"][:] = 37
            hm["capacity"][:] = 20.0
        cost = synthetic_tariff(96)[:T] if T != 24 else synthetic_tariff(24)
        rng = np.random.default_rng(T)
        p_est, p_sch = rng.uniform(0, 8, (H, T)), rng.uniform(0, 8, (H, T))
        gamma = rng.standard_normal((H, T))
        with gpu_lib.Solver([H], T) as s:
            s.set_homes(**hm)
            s.set_tariff(cost)
            g, p = s.home_step(p_est, p_sch, gamma, kappa=5.0)
        for i in range(H):
            ev = {} if not hm["has_ev"][i] else dict(rating=hm["rating"][i], capacity=hm["capacity"][i],
                                                     initial=hm["initial"][i], start=hm["start"][i], end=hm["end"][i])
            po, so, go = O.home_subproblem(cost, hm["load"][i], ev, p_est[i], p_sch[i], gamma[i], 5.0)
            assert np.array_equal(p[i], po), f"home {i} T={T}"
            assert np.array_equal(g[i], go)


def test_home_step_ties_pick_earliest_hour(gpu_lib):
    T, H = 24, 40
    load = np.full((H, T), 1.846)
    cost = np.full(T, 0.0951)
    hm = dict(load=load, has_ev=np.ones(H, np.uint8), rating=np.full(H, 4.8), capacity=np.full(H, 20.0),
              initial=np.full(H, 0.2), start=np.full(H, 11, np.int32), end=np.full(H, 23, np.int32))
    z = np.zeros((H, T))
    with gpu_lib.Solver([H], T) as s:
        s.set_homes(**hm)
        s.set_tariff(cost)
        g, p = s.home_step(z, z, z)
    assert (np.nonzero(p[0])[0] == [11, 12, 13]).all()
    assert np.array_equal(p, np.tile(p[0], (H, 1)))


def test_home_step_infeasible_is_an_error(gpu_lib):
    T, H = 24, 4
    hm = dict(load=np.ones((H, T)), has_ev=np.ones(H, np.uint8), rating=np.full(H, 4.8),
              capacity=np.full(H, 20.0), initial=np.full(H, 0.2), start=np.full(H, 11, np.int32),
              end=np.full(H, 13, np.int32))          # 2-hour window, 3 hours needed
    z = np.zeros((H, T))
    with gpu_lib.Solver([H], T) as s:
        s.set_homes(**hm)
        s.set_tariff(np.ones(T))
        with pytest.raises(gpu_lib.RevsError) as e:
            s.home_step(z, z, z)
        assert e.value.code == 3


# ----------------------------------------------------------------- other communities / adoption / rating (BASELINE config 2)
@pytest.mark.parametrize("com", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("adoption", [30, 60, 90])
@pytest.mark.parametrize("rating", [3600, 4800])
def test_sweep_points_match_oracle(gpu_lib, com, adoption, rating):
    """BASELINE.json config 2, all 30 points of the community x adoption x rating sweep on the
    reference's feeder: the distributed schedule equals the oracle's, charging hours bit for bit
    (hour costs are compared on the 2^-20 grid of oracle TIE_GRID, so the ~1e-12 differences of the
    two QP solvers cannot flip a tie -- in round 1 community 3 ended with 1-2 homes on another hour)."""
    from conftest import INPUT
    from revs_admm_b200.lpsolver import solve_ADMM
    from revs_admm_b200.revs_fixture import REVS
    fx = REVS(data_path=INPUT, out_path="/tmp/revs_out", grb_path="/tmp/revs_grb", fig_path="/tmp/revs_fig",
              regionID=121, networkID=121144, comunityID=com, optimizer_mode="distributed")
    tariff, homes, dist, saved = fx.read_inputs(adoption=adoption, rating=rating, seed=1234)
    kw = dict(kappa=5.0, iter_max=15, vset=1.03, vlow=0.95, vhigh=1.05)
    diff, P, S, C = solve_ADMM(homes, dist, tariff, None, **kw)
    do, Po, So, Co = O.solve_ADMM(homes, dist, tariff, None, **kw)
    assert len(saved["ev_homes"]) == int(adoption * 1e-2 * len(saved["community"]))
    assert all(np.array_equal(S[h], So[h]) for h in So)
    assert max(np.abs(P[h] - Po[h]).max() for h in Po) <= 1e-4
    assert max(abs(diff[k][h] - do[k][h]) for k in do for h in do[k]) <= 1e-7
    assert max(np.abs(C[h] - Co[h]).max() for h in Co) <= 1e-12


# ----------------------------------------------------------------- individual optimum
def test_individual_matches_oracle_and_golden_objective(gpu_lib, case121144, golden):
    from revs_admm_b200.lpsolver import solve_residences
    homes, tariff = case121144["homes"], case121144["tariff"]
    Pev, soc, Pres = solve_residences(tariff, homes)
    ev_ids = golden["individual_ev_ids"]
    c = np.asarray(tariff)
    for k, h in enumerate(ev_ids):
        h = int(h)
        po, so, go = O.solve_residence(tariff, homes[h])
        assert np.array_equal(Pev[h], po)
        assert np.allclose(soc[h], so, atol=1e-15)
        # the reference's own result: same objective (hours may differ where the tariff ties)
        gold_p, gold_s = golden["individual_P_ev"][k], golden["individual_SOC"][k]
        obj = 0.01 * c @ Pres[h] + 0.99 * (1 - soc[h][-1])
        load = Pres[h] - Pev[h]
        obj_gold = 0.01 * c @ (load + gold_p) + 0.99 * (1 - gold_s[-1])
        assert abs(obj - obj_gold) <= 1e-6 * abs(obj_gold)


@pytest.mark.parametrize("which", ["individual70", "individual3600"])
def test_individual_matches_other_reference_runs(gpu_lib, which, case_adopt70, case_rating3600, golden):
    """Device individual optimum against the two further result files of the reference
    (70 % adoption; 3600 W chargers): identical to the oracle, objective equal to the reference's."""
    from revs_admm_b200.lpsolver import solve_residences
    case = case_adopt70 if which == "individual70" else case_rating3600
    homes, tariff = case["homes"], case["tariff"]
    Pev, soc, Pres = solve_residences(tariff, homes)
    c = np.asarray(tariff)
    for k, h in enumerate(golden[f"{which}_ev_ids"]):
        h = int(h)
        po, so, go = O.solve_residence(tariff, homes[h])
        assert np.array_equal(Pev[h], po)
        gold_p, gold_s = golden[f"{which}_P_ev"][k], golden[f"{which}_SOC"][k]
        load = Pres[h] - Pev[h]
        obj = 0.01 * c @ Pres[h] + 0.99 * (1 - soc[h][-1])
        obj_gold = 0.01 * c @ (load + gold_p) + 0.99 * (1 - gold_s[-1])
        assert abs(obj - obj_gold) <= 1e-9 * abs(obj_gold)


# ----------------------------------------------------------------- utility step
def _rand_state(H, T, load, seed):
    rng = np.random.default_rng(seed)
    p_sch = load + 4.8 * (rng.random((H, T)) < 0.15)
    p_est = np.maximum(p_sch - rng.uniform(0, 1, (H, T)), 0)
    gamma = rng.standard_normal((H, T)) * 0.5
    return p_est, p_sch, gamma


def test_utility_step_real_feeder(gpu_lib, case121144):
    from revs_admm_b200.feeder import tree_from_graph
    dist, homes = case121144["dist"], case121144["homes"]
    tree = tree_from_graph(dist)
    res, Rres = O.residence_block(dist)
    assert res == tree.res_ids
    a = _arrays(homes, res)
    H, T = a["load"].shape
    p_est, p_sch, gamma = _rand_state(H, T, a["load"], 1)
    with gpu_lib.Solver([H], T) as s:
        s.set_feeder_tree(0, tree.parent, tree.r, tree.res_node)
        g, lam = s.utility_step(p_est, p_sch, gamma, kappa=5.0, vset=1.03, vlow=0.95, vhigh=1.05)
        st = s.stats()
    go, lo, _ = O.utility_subproblem(Rres, p_est, p_sch, gamma, 5.0, 1.03, 0.95, 1.05)
    assert np.abs(g - go).max() <= TOL_KW * 1e-2
    u = 1.05 ** 2 - 1.03 ** 2
    assert (Rres @ g).max() <= u + 1e-9
    assert g.min() >= 0.0
    # (the unsplit feeder has 1126 residences: it runs on the tree-Newton path, which needs no contraction)
    assert st["qp_newton_iterations"] > 0


def test_utility_step_multi_feeder_synthetic_tight(gpu_lib):
    from revs_admm_b200.feeder import synthetic_feeder, synthetic_homes
    sizes, T = [37, 150, 64], 24
    trees = [synthetic_feeder(n, seed=i, r_secondary=2e-3) for i, n in enumerate(sizes)]
    H = sum(sizes)
    hm = synthetic_homes(H, T, seed=3)
    p_est, p_sch, gamma = _rand_state(H, T, hm["load"], 5)
    vset, vhigh = 1.0, 1.01                      # tight: many rows active
    with gpu_lib.Solver(sizes, T) as s:
        for f, t in enumerate(trees):
            s.set_feeder_tree(f, t.parent, t.r, t.res_node)
        g, lam = s.utility_step(p_est, p_sch, gamma, kappa=5.0, vset=vset, vlow=0.9, vhigh=vhigh)
    off = np.concatenate([[0], np.cumsum(sizes)])
    for f, t in enumerate(trees):
        R = O.rmat_from_tree(t.parent, t.r)[np.ix_(t.res_node, t.res_node)]
        sl = slice(off[f], off[f + 1])
        go, _, _ = O.utility_subproblem(R, p_est[sl], p_sch[sl], gamma[sl], 5.0, vset, 0.9, vhigh)
        assert np.abs(g[sl] - go).max() <= TOL_KW * 1e-2


# ----------------------------------------------------------------- the whole loop
def test_admm_real_feeder_matches_oracle(gpu_lib, case121144, golden):
    """configs[0] of BASELINE.json: 121144 / Com-2 / 90 % / 4800 W, 15 iterations."""
    from revs_admm_b200.lpsolver import solve_ADMM
    homes, tariff, dist = case121144["homes"], case121144["tariff"], case121144["dist"]
    diff, P, S, C, stats = solve_ADMM(homes, dist, tariff, None, kappa=5.0, iter_max=15,
                                      vset=1.03, vlow=0.95, vhigh=1.05, return_stats=True)
    do, Po, So, Co = O.solve_ADMM(homes, dist, tariff, None, kappa=5.0, iter_max=15,
                                  vset=1.03, vlow=0.95, vhigh=1.05)
    res = list(Po)
    assert stats["admm_iterations"] == 15 and stats["kernel_launches"] > 45
    for h in res:
        assert np.array_equal(S[h], So[h]), f"charging hours differ at home {h}"
        assert np.abs(P[h] - Po[h]).max() <= TOL_KW
        assert np.allclose(C[h], Co[h], atol=1e-12)
    for k in range(1, 16):
        d = np.array([diff[k][h] for h in res])
        dref = np.array([do[k][h] for h in res])
        assert np.abs(d - dref).max() <= 1e-7, f"iteration {k}"
    # and the reference's own file where it is a function of the inputs: iteration 1
    ev_ids = [int(h) for h in golden["distributed_ev_ids"]]
    d1 = np.array([diff[1][h] for h in ev_ids])
    assert np.abs(d1 - golden["distributed_diff"][:, 0]).max() <= 1e-12
    # objective (tariff cost of the schedule) rel 1e-6
    c = np.asarray(tariff)
    cost = sum(c @ P[h] for h in res)
    cost_o = sum(c @ Po[h] for h in res)
    assert abs(cost - cost_o) <= 1e-6 * abs(cost_o)
    # voltages of the final schedule, GPU reliability check vs oracle
    from revs_admm_b200.lpsolver import compute_voltage, compute_flows
    V = compute_voltage(dist, P, vset=1.03)
    Vo = O.compute_voltage(dist, Po, vset=1.03)
    assert max(np.abs(np.asarray(V[n]) - Vo[n]).max() for n in Vo) <= TOL_PU
    Fl = compute_flows(dist, P)
    Fo = O.compute_flows(dist, Po)
    assert max(np.abs(np.asarray(Fl[e]) - Fo[e]).max() for e in Fo) <= 1e-6


def test_admm_multi_feeder_synthetic_96(gpu_lib):
    """Shape of configs[2..4]: several feeders, 96 quarter-hour steps, tight limits."""
    from revs_admm_b200.feeder import synthetic_feeder, synthetic_homes, synthetic_tariff
    sizes, T = [90, 61, 130], 96
    trees = [synthetic_feeder(n, seed=10 + i, r_secondary=1e-3) for i, n in enumerate(sizes)]
    H = sum(sizes)
    hm = synthetic_homes(H, T, seed=11)
    cost = synthetic_tariff(T)
    kw = dict(kappa=5.0, iter_max=6, vset=1.0, vlow=0.95, vhigh=1.02)
    with gpu_lib.Solver(sizes, T) as s:
        s.set_feeder_trees(trees)                      # one upload + one kernel for all feeders
        s.set_homes(**hm)
        s.set_tariff(cost)
        done = s.solve_admm(**kw)
        out = s.results(done)
        P_est, Gam = s.estimate()
        for f, t in enumerate(trees):                  # same blocks as the per-feeder entry point
            drop = s.reliability(f, 2, t.res_node, P=np.eye(len(t.res_node), T))
    Rb = [O.rmat_from_tree(t.parent, t.r)[np.ix_(t.res_node, t.res_node)] for t in trees]
    ref = O.solve_ADMM_arrays(Rb, cost=cost, **_oracle_kwargs(hm), **kw)
    assert np.array_equal(out["P_ev"], ref["P_ev"])
    assert np.abs(out["P_sch"] - ref["P_sch"]).max() <= TOL_KW
    assert np.abs(P_est - ref["P_est"]).max() <= TOL_KW
    assert np.abs(Gam - ref["Gamma"]).max() <= 1e-4
    assert np.abs(out["diff"] - ref["diff"]).max() <= 1e-7
    assert np.allclose(out["SOC"], ref["SOC"], atol=1e-12)


def test_admm_early_stop_and_step_api(gpu_lib):
    from revs_admm_b200.feeder import synthetic_feeder, synthetic_homes, synthetic_tariff
    n, T = 50, 24
    t = synthetic_feeder(n, seed=2, r_secondary=1e-5)       # loose network: converges quickly
    hm = synthetic_homes(n, T, seed=2)
    with gpu_lib.Solver([n], T) as s:
        s.set_feeder_tree(0, t.parent, t.r, t.res_node)
        s.set_homes(**hm)
        s.set_tariff(synthetic_tariff(T))
        done = s.solve_admm(iter_max=40, tol=1e-6)
        assert done < 40
        st = s.stats()
        assert st["primal_residual"] < 1e-6 and st["dual_residual"] < 1e-6
        full = s.results(done)
        s.admm_begin(iter_max=done)
        for _ in range(done):
            sums = s.admm_step()
        assert sums[2] == n * T
        again = s.results(done)
    assert np.array_equal(full["P_sch"], again["P_sch"])
    assert np.array_equal(full["diff"], again["diff"])


# ----------------------------------------------------------------- screening contraction
@pytest.mark.parametrize("impl", [0, 1])
@pytest.mark.parametrize("M,K,T", [(128, 64, 96), (1008, 1008, 96), (130, 100, 24), (77, 333, 5), (300, 48, 96)])
def test_screen_contract_bound(gpu_lib, impl, M, K, T):
    """BF16 screening product: rigorous one-sided bound v <= 1.0099 v~ on non-negative data,
    for the mma.sync kernel (impl 0) and the tcgen05/TMEM/TMA kernel (impl 1)."""
    rng = np.random.default_rng(M + K + T)
    A = rng.uniform(0, 2e-2, (M, K)) * (rng.random((M, K)) < 0.7)
    B = rng.uniform(0, 8, (K, T))
    C = gpu_lib.screen_contract(A, B, impl=impl)
    ref = A @ B
    assert C.shape == ref.shape
    rel = np.abs(C - ref) / np.maximum(ref, 1e-300)
    assert rel[ref > 0].max() <= 9.9e-3
    assert (ref <= 1.0099 * C + 1e-30).all()


def test_screen_impls_agree_in_the_loop(gpu_lib):
    from revs_admm_b200.feeder import synthetic_feeder, synthetic_homes, synthetic_tariff
    sizes, T = [130, 77, 201], 96
    trees = [synthetic_feeder(n, seed=30 + i, r_secondary=1e-3) for i, n in enumerate(sizes)]
    hm = synthetic_homes(sum(sizes), T, seed=31)
    outs = []
    for impl in (0, 1):
        with gpu_lib.Solver(sizes, T) as s:
            s.set_option("screen_impl", impl)
            s.set_feeder_trees(trees)
            s.set_homes(**hm)
            s.set_tariff(synthetic_tariff(T))
            done = s.solve_admm(kappa=5.0, iter_max=5, vset=1.0, vlow=0.95, vhigh=1.015)
            outs.append(s.results(done))
    for k in ("P_sch", "P_ev", "SOC", "diff"):
        assert np.array_equal(outs[0][k], outs[1][k]), k


# ----------------------------------------------------------------- centralized schedule
def test_centralized_matches_reference_file(gpu_lib, case121144, golden):
    """solve_central (lpsolver.py:463-502) through REVS.get_centralized_optimal against the reference's own
    result file out/121144-com2/centralized/adopt90-rating4800-seed1234.txt: residence profiles, charger
    profiles and SOC profiles equal (the reference's program has no final-SOC row: no charging)."""
    fx, homes, tariff, dist = case121144["fx"], case121144["homes"], case121144["tariff"], case121144["dist"]
    Pres, Pev, soc = fx.get_centralized_optimal(tariff, homes, dist, save=False, v0=1.03, vmin=0.90, vmax=1.05)
    res = [int(h) for h in golden["centralized_res_ids"]]
    assert list(Pres) == res
    for i, h in enumerate(res):
        assert np.abs(np.asarray(Pres[h]) - golden["centralized_P_res"][i]).max() <= 1e-12
    for k, h in enumerate(golden["centralized_ev_ids"]):
        assert np.array_equal(Pev[int(h)], golden["centralized_P_ev"][k])
        assert np.array_equal(soc[int(h)], golden["centralized_SOC"][k])
    # the voltage rows decide feasibility: with vmin just below v0 the base load alone violates them
    from revs_admm_b200.lpsolver import solve_central
    with pytest.raises(RuntimeError, match="No solution found"):
        solve_central(tariff, homes, dist, None, 1.03, 1.0299, 1.05)

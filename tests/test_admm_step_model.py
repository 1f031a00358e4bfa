"""CPU checks of the one-iteration model (tests/admm_step_ref.py) before it judges the device: the projection
certificate accepts the oracle's projections -- duplicate binding rows and all-negative targets included -- and
rejects the same point moved by 1e-7 kW; next_target and dual_update keep the kernels' operation order."""
import math
from fractions import Fraction

import numpy as np
import pytest

import admm_step_ref as AR
import revs_oracle as O
from revs_admm_b200.feeder import synthetic_feeder

U = 1.02 ** 2 - 1.0


def _project(R, z, u):
    g = np.empty_like(z)
    for t in range(z.shape[1]):
        g[:, t] = O.project_voltage(z[:, t], R, u)[0]
    return g


def _synthetic_zone():
    """30 residences of a synthetic feeder, 8 columns of targets from -1 to 6 kW; column 0 is <= 0 everywhere."""
    t = synthetic_feeder(30, seed=4, r_secondary=2e-3)
    R = O.rmat_from_tree(t.parent, t.r)[np.ix_(t.res_node, t.res_node)]
    z = np.random.default_rng(4).uniform(-1.0, 6.0, (30, 8))
    z[:, 0] = -np.abs(z[:, 0])
    return R, z


def _shared_node_zone():
    """A chain 0 - 1 - 2 with branches: residences 0 and 1 on node 3, so rows 0 and 1 of R are identical, and they
    carry the largest resistance, so they bind first."""
    parent = np.array([-1, 0, 1, 2, 2, 1, 0])
    r = np.array([2.5e-4, 5e-4, 2.5e-4, 1.5e-3, 2.5e-4, 5e-4, 2.5e-4])
    res_node = np.array([3, 3, 4, 5, 6, 2, 4])
    R = O.rmat_from_tree(parent, r)[np.ix_(res_node, res_node)]
    z = np.random.default_rng(7).uniform(-1.5, 12.0, (len(res_node), 6))
    z[:2] += 4.0                                      # the two residences of node 3 want the most
    return R, z


@pytest.mark.parametrize("zone", [_synthetic_zone, _shared_node_zone])
@pytest.mark.parametrize("use_lstsq", [True, False])
def test_certificate_accepts_the_oracle_projection(zone, use_lstsq):
    R, z = zone()
    g = _project(R, z, U)
    c = AR.certify_projection(R, z, g, U, use_lstsq=use_lstsq)
    assert c["ok"].all(), c["resid"]
    assert (c["rows"] > 0).sum() >= 3                  # rows bind in most columns
    if not use_lstsq:
        assert c["lp"] == (c["rows"] > 0).sum()
    if zone is _synthetic_zone:
        assert c["rows"][0] == 0 and not g[:, 0].any()    # z <= 0: g = 0, no row near u
    else:
        V = R @ g
        both = (V[0] >= U - 1e-9) & (V[1] >= U - 1e-9)
        assert np.array_equal(R[0], R[1]) and both.any()  # the duplicate rows bind together


def _column_with_everything(R, z, g):
    """A column with a binding row, a free home and a home at zero whose target is negative."""
    V = R @ g
    for t in range(z.shape[1]):
        if (V[:, t] >= U - 1e-9).any() and (g[:, t] > 0).any() and ((g[:, t] == 0) & (z[:, t] < -1e-3)).any():
            return t
    raise AssertionError("no suitable column")


@pytest.mark.parametrize("zone", [_synthetic_zone, _shared_node_zone])
@pytest.mark.parametrize("move", ["free", "zero", "row"])
@pytest.mark.parametrize("use_lstsq", [True, False])
def test_certificate_rejects_a_moved_point(zone, move, use_lstsq):
    """1e-7 kW on one home: a free one, one at zero (g_j = 1e-7), or the free home with the largest entry in a binding
    row, which pushes that row past u.  The homes are picked so that every row moves by less than tol = 1e-9:
    only the multiplier conditions can reject the point."""
    R, z = zone()
    g = _project(R, z, U)
    t = _column_with_everything(R, z, g)
    col = g[:, t]
    V = R @ col
    small = R.max(axis=0) < 9e-3                      # 1e-7 kW on home j moves no row by more than 9e-10
    if move == "free":
        j = int(np.nonzero(small & (col > 0))[0][0])
    elif move == "zero":
        j = int(np.nonzero(small & (col == 0) & (z[:, t] < -1e-3))[0][0])
    else:
        i = int(np.argmax(V))
        j = int(np.argmax(np.where(small & (col > 0), R[i], -1.0)))
        assert V[i] >= U - 1e-12 and R[i, j] > 0
    bad = g.copy()
    bad[j, t] += 1e-7
    assert np.abs(R @ bad[:, t] - V).max() < 1e-9
    c = AR.certify_projection(R, z, bad, U, use_lstsq=use_lstsq)
    assert not c["ok"][t] and c["resid"][t] > 1e-9
    others = np.arange(z.shape[1]) != t
    assert c["ok"][others].all()


def test_certificate_rejects_infeasible_and_negative_points():
    R, z = _synthetic_zone()
    g = _project(R, z, U)
    c = AR.certify_projection(R, z, g * (1.0 + 1e-6), U)          # every binding row past u by ~4e-8
    assert not c["ok"][c["rows"] > 0].any()
    neg = g.copy()
    neg[0, 0] = -1e-300
    assert not AR.certify_projection(R, z, neg, U)["ok"][0]
    off = g.copy()
    off[3, 0] = 1e-11                                              # no candidate row: g must be [z]_+ to 1e-12
    assert not AR.certify_projection(R, z, off, U)["ok"][0]


def test_next_target_and_dual_update_keep_the_kernel_order():
    """Every element against the kernels' expression in scalar arithmetic: 0 ulp.  diff against the exact sum of
    squares: within one rounding of the sqrt argument."""
    rng = np.random.default_rng(3)
    H, T, kappa = 5, 37, 3.7
    P_est, P_sch, Gamma = rng.uniform(0, 6, (H, T)), rng.uniform(0, 6, (H, T)), rng.normal(0, 3, (H, T))
    z = AR.next_target(P_est, P_sch, Gamma, kappa)
    G1, diff = AR.dual_update(Gamma, P_est, P_sch, kappa)
    hk = 0.5 * kappa
    for h in range(H):
        for t in range(T):
            e, s, gm = float(P_est[h, t]), float(P_sch[h, t]), float(Gamma[h, t])
            assert z[h, t] == (e + s) * 0.5 - gm / kappa
            assert G1[h, t] == gm + hk * (e - s)
        exact = sum(Fraction(float(c)) ** 2 for c in P_est[h] - P_sch[h])
        want = math.sqrt(float(exact)) / T
        assert abs(diff[h] - want) <= 2.3e-16 * want
    assert not np.array_equal(z, (P_est + P_sch) * 0.5 - Gamma * (1.0 / kappa))    # the order does matter


def test_certificate_accepts_projections_that_need_the_lp_at_its_bound():
    """Iteration 3 of the tree-Newton ADMM case with shared nodes and daisy chains (test_gpu_admm_steps, newton_odd):
    the LP's multipliers for columns with hundreds of candidate rows sit on the bound of the homes at zero, and were
    rejected by rounding (residual 1.000005e-9) when that bound was the acceptance tolerance itself."""
    from test_gpu_newton_shapes import odd_wide
    from revs_admm_b200.feeder import synthetic_homes, synthetic_tariff
    tr = odd_wide()
    T = 24
    hm = synthetic_homes(tr.n_res, T, seed=tr.n_res)
    kw = dict(kappa=5.0, vset=1.0, vlow=0.95, vhigh=1.02)
    R = O.rmat_from_tree(tr.parent, tr.r)[np.ix_(tr.res_node, tr.res_node)]
    u = kw["vhigh"] ** 2 - kw["vset"] ** 2
    h = O.solve_ADMM_arrays([R], load=hm["load"], cost=synthetic_tariff(T), ev_mask=hm["has_ev"].astype(bool),
                            rating=hm["rating"], capacity=hm["capacity"], initial=hm["initial"], start=hm["start"],
                            end=hm["end"], iter_max=2, return_history=True, **kw)["history"]
    z = AR.next_target(*h[1], kw["kappa"])[:, [21, 22]]           # the two columns of iteration 3 that were rejected
    g = np.stack([O.project_voltage(z[:, j], R, u)[0] for j in range(2)], axis=1)
    c = AR.certify_projection(R, z, g, u)
    assert c["ok"].all() and c["lp"] >= 1, (np.nonzero(~c["ok"])[0], c["resid"].max(), c["lp"])

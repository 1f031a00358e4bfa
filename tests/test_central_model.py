"""CPU: the numpy model of the bracket of the centralized optimum (tests/central_ref.py) against the exact MILP optimum
of every zone (scipy.optimize.milp): LB <= optimum <= UB, the kept schedule meets every row (dense sensitivity
matrix) and every home's windows, LB is at least bench.objective_check's bound, loose limits give status 0 and a
base load that violates a row gives status 3."""
import numpy as np
import pytest
from scipy.optimize import Bounds, LinearConstraint, milp
from scipy.sparse import csr_matrix, vstack

import bench
import central_ref as CR
import network_ref as NR
from revs_admm_b200.feeder import FeederTree, population, synthetic_feeder, synthetic_homes, synthetic_tariff

REL = 1e-9


def _zones(seed):
    """Small zones (at most 40 residences), several residences on one node and nodes without any, a one-node zone."""
    rng = np.random.default_rng(seed)
    out = []
    for n in (12, 25, 40):
        t = synthetic_feeder(n, seed=seed + n, laterals=2, r_secondary=3e-4)
        res = t.res_node.copy()
        res[1::4] = res[0]
        res[2::7] = rng.integers(0, t.n_nodes - n, len(res[2::7]))
        out.append(FeederTree(parent=t.parent, r=t.r, res_node=res.astype(np.int32)))
    out.insert(1, FeederTree(parent=np.array([-1], np.int32), r=np.array([1e-3]), res_node=np.zeros(4, np.int32)))
    return out


def _homes(H, T, seed):
    hm = synthetic_homes(H, T, seed=seed)
    rng = np.random.default_rng(seed)
    hm["initial"] = rng.uniform(0.05, 0.4, H)             # various SOC windows: some homes may charge optional hours
    sph = max(1, T // 24)
    hm["start"] = np.minimum(rng.integers(8, 13, H) * sph, T - 1).astype(np.int32)
    hm["end"] = np.minimum(hm["start"] + rng.integers(9, 14, H) * sph, T).astype(np.int32)
    k0 = np.maximum(1, ((hm["end"] - hm["start"]) * rng.uniform(0.2, 0.6, H)).astype(int))
    hm["capacity"] = hm["rating"] * (k0 - 0.05) / (0.9 - hm["initial"])     # n_min = k0 fits the window
    return hm


def _split(zones, hm):
    off = 0
    for tr in zones:
        yield tr, {k: np.asarray(v)[off:off + tr.n_res] for k, v in hm.items()}
        off += tr.n_res


def _u_between(zones, hm, cost, frac):
    """u between the largest drop of the base load (frac 0) and that of every home's cheapest hours (frac 1)."""
    base = NR.network_check(zones, hm["load"])["drop"].max()
    cheap = np.concatenate([CR._Zone(tr, hz, cost).P(CR._Zone(tr, hz, cost).priced(np.zeros((tr.n_res, len(cost)))))
                            for tr, hz in _split(zones, hm)])
    top = NR.network_check(zones, cheap)["drop"].max()
    return float(base + frac * (top - base))


def _milp(tr, hz, cost, u):
    """Exact optimum of the zone's centralized problem (None when infeasible)."""
    Z = CR._Zone(tr, hz, cost)
    Rres = tr.rmat()[np.ix_(Z.res, Z.res)]
    idx = np.argwhere(Z.win)
    c = Z.rating[idx[:, 0]] * Z.cost[idx[:, 1]]
    base = Rres @ Z.load - u                               # [n, T]
    blocks, b = [], []
    for t in range(len(Z.cost)):
        k = np.nonzero(idx[:, 1] == t)[0]
        A = np.zeros((tr.n_res, len(idx)))
        A[:, k] = Rres[:, idx[k, 0]] * Z.rating[idx[k, 0]]
        blocks.append(csr_matrix(A))
        b.append(-base[:, t])
    hh = np.unique(idx[:, 0]) if len(idx) else np.zeros(0, int)
    cons = [LinearConstraint(vstack(blocks), -np.inf, np.concatenate(b))]
    if len(hh):
        cons.append(LinearConstraint(csr_matrix((np.ones(len(idx)), (np.searchsorted(hh, idx[:, 0]), np.arange(len(idx)))),
                                                shape=(len(hh), len(idx))), Z.nmin[hh], Z.nmax[hh]))
    if len(idx) == 0:
        return float((Z.load @ Z.cost).sum()) if (base <= 0).all() else None
    r = milp(c, constraints=cons, integrality=np.ones(len(idx)), bounds=Bounds(0, 1))
    return None if r.status == 2 else float(r.fun + (Z.load @ Z.cost).sum())


def _check_zone(tr, hz, cost, u, P, bits, bounds, info, opt):
    lb, ub = bounds
    st = info[0]
    Z = CR._Zone(tr, hz, cost)
    if st in (0, 1):
        assert opt is not None
        assert lb <= opt + REL * abs(opt) and opt <= ub + REL * abs(opt)
        Rres = tr.rmat()[np.ix_(Z.res, Z.res)]
        assert (Rres @ P - u <= 1e-9 + 1e-12).all()
        cnt = bits.sum(axis=1)
        assert not (bits & ~Z.win).any() and (cnt >= Z.nmin).all() and (cnt <= Z.nmax).all()
        assert np.array_equal(P, Z.P(bits))
        assert float((P @ Z.cost).sum()) == pytest.approx(ub, rel=REL)
        if st == 0:
            assert lb == ub
    else:
        assert ub == np.inf
        if st == 3:
            assert opt is None
        elif opt is not None:
            assert lb <= opt + REL * abs(opt)
    _, lb0, _ = bench.objective_check([], hz, Z.cost, P, len(Z.cost))
    assert lb >= lb0 - REL * abs(lb0)


@pytest.mark.parametrize("frac", [0.3, 0.6])
def test_bracket_contains_the_optimum_on_small_zones(frac):
    T = 24
    zones = _zones(7)
    hm = _homes(sum(z.n_res for z in zones), T, 7)
    cost = synthetic_tariff(T)
    u = _u_between(zones, hm, cost, frac)
    out = CR.bracket(zones, hm, cost, vset=1.0, vhigh=np.sqrt(1.0 + u), iters=60)
    u = np.sqrt(1.0 + u) ** 2 - 1.0                      # the model's u, rounded as it rounds it
    st = out["zone_info"][:, 0]
    assert (st == 1).any() and (out["zone_info"][:, 1] > 0).any()
    off = 0
    for z, (tr, hz) in enumerate(_split(zones, hm)):
        s = slice(off, off + tr.n_res)
        off += tr.n_res
        _check_zone(tr, hz, cost, u, out["P_sch"][s], out["bits"][s], out["zone_bounds"][z], out["zone_info"][z],
                    _milp(tr, hz, cost, u))


def test_reference_shaped_zone():
    """Zone 3 of one reference-shaped feeder at the bench's limits (vset 1.03, vhigh 1.05)."""
    trees, hm, cost, sizes, T = population("refshape", 1, seed=0)
    tr, hz = list(_split(trees, hm))[3]
    out = CR.bracket([tr], hz, cost, vset=1.03, vhigh=1.05, iters=100)
    u = 1.05 * 1.05 - 1.03 * 1.03
    assert out["zone_info"][0, 0] == 1
    _check_zone(tr, hz, cost, u, out["P_sch"], out["bits"], out["zone_bounds"][0], out["zone_info"][0],
                _milp(tr, hz, cost, u))


def test_loose_limits_are_optimal():
    T = 24
    zones = _zones(4)
    hm = _homes(sum(z.n_res for z in zones), T, 4)
    cost = synthetic_tariff(T)
    out = CR.bracket(zones, hm, cost, vset=1.0, vhigh=1.5, iters=30)
    assert (out["zone_info"] == 0).all()
    u = 1.5 * 1.5 - 1.0
    for z, (tr, hz) in enumerate(_split(zones, hm)):
        lb, ub = out["zone_bounds"][z]
        assert lb == ub and ub == pytest.approx(_milp(tr, hz, cost, u), rel=REL)


def test_base_load_violation_is_certified_infeasible():
    T = 24
    zones = _zones(3)
    hm = _homes(sum(z.n_res for z in zones), T, 3)
    cost = synthetic_tariff(T)
    drop = NR.network_check(zones, hm["load"])["drop"]
    u = 0.95 * float(drop.max())
    out = CR.bracket(zones, hm, cost, vset=1.0, vhigh=np.sqrt(1.0 + u), iters=60)
    u = np.sqrt(1.0 + u) ** 2 - 1.0
    off = noff = 0
    for z, (tr, hz) in enumerate(_split(zones, hm)):
        base = drop[noff:noff + tr.n_nodes][tr.res_node] - u
        noff += tr.n_nodes
        if (base > 1e-9).any():
            assert out["zone_info"][z, 0] == 3 and out["zone_bounds"][z, 1] == np.inf
            assert _milp(tr, hz, cost, u) is None
        off += tr.n_res
    assert (out["zone_info"][:, 0] == 3).any()


def test_a_window_too_short_for_the_soc_target_is_refused():
    T = 24
    zones = _zones(2)[:1]
    hm = _homes(zones[0].n_res, T, 2)
    h = int(np.nonzero(hm["has_ev"])[0][0])
    hm["end"][h] = hm["start"][h] + 1
    hm["capacity"][h] = hm["rating"][h] * 2.5 / (0.9 - hm["initial"][h])     # n_min = 3 > 1 window hour
    with pytest.raises(ValueError):
        CR.bracket(zones, hm, synthetic_tariff(T))


def test_fsum_is_the_kernel_order():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((37, 29)) * 10.0 ** rng.integers(-8, 8, (37, 29))
    v = x.ravel()
    lanes = [0.0] * 256
    for j, a in enumerate(v):
        lanes[j % 256] = lanes[j % 256] + a
    for o in (16, 8, 4, 2, 1):
        lanes = [lanes[i] + lanes[i ^ o] for i in range(256)]
    s = lanes[0]
    for w in range(1, 8):
        s = s + lanes[32 * w]
    assert CR.fsum(x) == s

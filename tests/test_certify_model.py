"""CPU: the numpy model of the certificate of voltage infeasibility (tests/certify_ref.py).  Soundness against the exact
MILP of small zones (scipy.optimize.milp), the case the Lagrangian bound of central_bracket cannot see (LP relaxation
feasible, binary program infeasible), each kind of certificate on a hand-built zone, the rounding margin, the witness
of a reference-shaped zone rebuilt with the dense sensitivity matrix, and central_status."""
import numpy as np
import pytest
from scipy.optimize import linprog

import central_ref as CR
import certify_ref as CF
from revs_admm_b200 import central_status
from revs_admm_b200.feeder import FeederTree, population, synthetic_tariff
from test_central_model import _homes, _milp, _split, _u_between, _zones


def _vhigh(u):
    return float(np.sqrt(1.0 + u))


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_certified_zones_have_no_binary_schedule(seed):
    T = 24
    zones = _zones(seed)
    hm = _homes(sum(z.n_res for z in zones), T, seed)
    cost = synthetic_tariff(T)
    certified = infeasible = 0
    for frac in (0.0, 0.1, 0.25, 0.5):
        u = _u_between(zones, hm, cost, frac)
        got = CF.certify(zones, hm, vset=1.0, vhigh=_vhigh(u))["zone_cert"]
        uu = _vhigh(u) ** 2 - 1.0                 # the u the model used
        for (tr, hz), c in zip(_split(zones, hm), got):
            opt = _milp(tr, hz, cost, uu + 1e-9)
            infeasible += opt is None
            if c[0]:
                certified += 1
                assert opt is None, (frac, c)
                if c[0] == 2:
                    assert CF.recheck(tr, hz, c, vset=1.0, vhigh=_vhigh(u)) == c[3]
                else:
                    assert CF.recheck(tr, hz, c, vset=1.0, vhigh=_vhigh(u)) > 0
    assert certified > 0 and infeasible >= certified


def _one_node(n, r=0.5):
    """A zone of n residences on one node: R[i,h] = 2 r for every pair."""
    return FeederTree(parent=np.array([-1], np.int32), r=np.array([r]), res_node=np.zeros(n, np.int32))


def _hand_homes(n, T, start, end, nmin=1, load=None):
    """n EV homes of rating 1, SOC target nmin hours (n_min = n_max = nmin), window [start, end)."""
    return dict(load=np.zeros((n, T)) if load is None else load, has_ev=np.ones(n, np.uint8), rating=np.ones(n),
                capacity=np.full(n, nmin / 0.5), initial=np.full(n, 0.5),
                start=np.full(n, start, np.int32), end=np.full(n, end, np.int32))


def _lp_feasible(tr, hz, u, row_tol=1e-9):
    """The LP relaxation of the zone's program (e in [0, 1], n_min <= sum e over the window) has a solution."""
    Z = CR._Zone(tr, hz, np.zeros(hz["load"].shape[1]))
    R = tr.rmat()[np.ix_(Z.res, Z.res)]
    n, T = Z.load.shape
    A_ub, b_ub = [], []
    base = R @ Z.load - u
    for t in range(T):
        for i in range(n):
            row = np.zeros((n, T))
            row[:, t] = R[i] * Z.rating
            A_ub.append(row.ravel())
            b_ub.append(row_tol - base[i, t])
    for h in range(n):
        row = np.zeros((n, T))
        row[h] = -1.0
        A_ub.append(row.ravel())
        b_ub.append(-Z.nmin[h])
    bounds = [(0.0, 1.0 if Z.win[h, t] else 0.0) for h in range(n) for t in range(T)]
    return linprog(np.zeros(n * T), A_ub=np.array(A_ub), b_ub=np.array(b_ub), bounds=bounds).status == 0


def test_lp_feasible_but_no_binary_schedule():
    """Three homes, one charge each, two steps, room for one and a half charges per step: the LP relaxation charges
    every home half an hour at each step, the binary program has room for two charges only.  The Lagrangian bound
    equals the LP bound, so central_bracket leaves the zone open (status 2); the counting certificate proves it."""
    T, u = 4, 1.6
    tr, hz = _one_node(3), _hand_homes(3, T, 1, 3)
    cost = synthetic_tariff(T)
    assert _lp_feasible(tr, hz, u)
    assert _milp(tr, hz, cost, u + 1e-9) is None
    c = CF.certify([tr], hz, vset=1.0, vhigh=_vhigh(u))["zone_cert"][0]
    assert c.tolist() == [2, 0, 3, 1]              # S_3: two charges fit, three are needed
    assert CR.bracket([tr], hz, cost, vset=1.0, vhigh=_vhigh(u), iters=100)["zone_info"][0, 0] == 2


def test_kind_1_base_load():
    T, u = 6, 1.6
    load = np.zeros((3, T))
    load[2, 4] = 1.0
    load[1, 3] = 1.7                               # D0 = 1.7 at every residence of the node, step 3 (the worst)
    load[0, 5] = 1.7
    c = CF.certify([_one_node(3)], _hand_homes(3, T, 0, 6, load=load), vset=1.0, vhigh=_vhigh(u))["zone_cert"][0]
    assert c.tolist() == [1, 0, 3, 0]


def test_kind_2_one_home():
    """One home needs both hours of its window, and the base load leaves room for its charge at one of them only."""
    T, u = 4, 1.6
    load = np.zeros((2, T))
    load[1, 2] = 1.1                               # slack 0.5 < rating at step 2
    hz = _hand_homes(2, T, 1, 3, nmin=2, load=load)
    hz["has_ev"] = np.array([1, 0], np.uint8)
    c = CF.certify([_one_node(2)], hz, vset=1.0, vhigh=_vhigh(u))["zone_cert"][0]
    assert c.tolist() == [2, 0, 1, 1]
    assert _milp(_one_node(2), hz, synthetic_tariff(T), u + 1e-9) is None


def test_kind_2_needs_several_homes():
    """Five homes, one charge each, three steps, room for one charge per step: no one, two or three homes are short of
    room, four are one charge short and all five two."""
    T, u = 5, 1.6
    tr, hz = _one_node(5), _hand_homes(5, T, 1, 4)
    c = CF.certify([tr], hz, vset=1.0, vhigh=_vhigh(u))["zone_cert"][0]
    assert c[0] == 2 and c[2] >= 2 and c.tolist() == [2, 0, 5, 2]
    assert CF.recheck(tr, hz, c, vset=1.0, vhigh=_vhigh(u)) == 2


def test_margin_resolves_in_favour_of_fits(monkeypatch):
    """Four homes, one charge each, two steps; two charges exceed u + row_tol by 5e-13 pu^2 at every step.  Inside the
    1e-12 margin they fit, so the zone is not certified; without the margin it would be."""
    T, vhigh, tol = 4, _vhigh(1.6), 1e-9
    u = vhigh * vhigh - 1.0
    load = np.zeros((4, T))
    load[0, 1:3] = u - 2.0 + tol + 5e-13
    tr, hz = _one_node(4), _hand_homes(4, T, 1, 3, load=load)
    assert CF.certify([tr], hz, vset=1.0, vhigh=vhigh, row_tol=tol)["zone_cert"][0].tolist() == [0, -1, -1, 0]
    monkeypatch.setattr(CF, "MARGIN", 0.0)
    assert CF.certify([tr], hz, vset=1.0, vhigh=vhigh, row_tol=tol)["zone_cert"][0, 0] == 2


def test_reference_zone_6():
    """Zone 6 of the first two reference-shaped feeders at the bench's limits: the bracket leaves it open, and four
    homes on residence 121's row are ten charges short of their SOC targets."""
    trees, hm, cost, sizes, T = population("refshape", 2, seed=0)
    got = CF.certify(trees, hm, vset=1.03, vhigh=1.05)["zone_cert"]
    assert got[6].tolist() == [2, 121, 4, 10]
    assert (got[np.arange(len(trees)) != 6, 0] == 0).all()
    tr, hz = list(_split(trees, hm))[6]
    assert CF.recheck(tr, hz, got[6], vset=1.03, vhigh=1.05) == 10


def test_errors():
    T = 4
    hz = _hand_homes(2, T, 1, 3, nmin=3)           # n_min 3 > 2 window hours
    with pytest.raises(ValueError, match="window"):
        CF.certify([_one_node(2)], hz)
    hz = _hand_homes(2, T, 1, 3)
    hz["rating"] = np.array([1.0, np.inf])
    with pytest.raises(ValueError, match="rating"):
        CF.certify([_one_node(2)], hz)


def test_central_status():
    info = np.array([[0, 0, 0], [1, 5, 3], [2, 100, 0], [2, 100, 0], [3, 40, 0]], np.int32)
    cert = np.array([[0, -1, -1, 0], [0, -1, -1, 0], [2, 4, 3, 1], [0, -1, -1, 0], [1, 0, 7, 0]], np.int32)
    assert central_status(info, cert).tolist() == [0, 1, 3, 2, 3]
    assert info[:, 0].tolist() == [0, 1, 2, 2, 3]
    cert[1, 0] = 2
    with pytest.raises(ValueError, match=r"\[1\]"):
        central_status(info, cert)

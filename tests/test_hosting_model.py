"""CPU checks of the hosting capacity model (tests/hosting_ref.py): it equals the definition min_i sigma_i / R[i,h] bit
for bit, the dense R of FeederTree.rmat() to rounding, the thermal terms' path minimum and the dense R 1; and adding a
home's capacity keeps every row and rated edge of its zone within its limit, while a little more breaks one."""
import numpy as np
import pytest

import hosting_ref as HR
import network_ref as NR
from revs_admm_b200.feeder import FeederTree, population, synthetic_feeder
from test_network_model import _zones

VSET, VHIGH, TOL = 1.0, 1.05, 1e-9
UR = (VHIGH * VHIGH - VSET * VSET) + TOL


def _cases():
    """(zones, P): mixed synthetic zones at two load levels (the heavier one violates rows) and reference-shaped zones."""
    out = []
    for seed, hi in ((1, 2.0), (2, 60.0)):
        zones = _zones(seed)
        rng = np.random.default_rng(seed)
        out.append((zones, rng.uniform(0.0, hi, (sum(z.n_res for z in zones), 7))))
    trees, hm, cost, sizes, T = population("refshape", 1, seed=0)
    trees = trees[:6]
    H = sum(t.n_res for t in trees)
    out.append((trees, hm["load"][:H] * 4.0))
    return out


def _each_zone(zones, P):
    off = 0
    for tr in zones:
        yield tr, P[off:off + tr.n_res]
        off += tr.n_res


@pytest.mark.parametrize("case", range(3))
def test_equals_the_definition_bit_for_bit(case):
    zones, P = _cases()[case]
    saw_zero = saw_pos = False
    for tr, Pz in _each_zone(zones, P):
        z = HR.zone_hosting(tr, Pz, UR)
        brute = HR.brute_voltage(tr, Pz, UR)
        assert np.array_equal(z["cap"], brute)
        saw_zero |= bool((brute == 0.0).any())
        saw_pos |= bool(((brute > 0.0) & np.isfinite(brute)).any())
    assert saw_pos and (saw_zero or case != 1)


@pytest.mark.parametrize("case", range(3))
def test_agrees_with_the_dense_sensitivity(case):
    zones, P = _cases()[case]
    for tr, Pz in _each_zone(zones, P):
        res = np.asarray(tr.res_node, dtype=np.int64)
        R = tr.rmat()[np.ix_(res, res)]
        sigma = UR - R @ Pz
        cap = HR.zone_hosting(tr, Pz, UR)["cap"]
        for h in range(tr.n_res):
            k = R[:, h] > 0.0
            if not k.any():
                assert np.isinf(cap[h]).all()
                continue
            ref = (sigma[k] / R[k, h][:, None]).min(axis=0)
            ref = np.where(ref > 0.0, ref, 0.0)
            assert np.allclose(cap[h], ref, rtol=1e-12, atol=1e-12 * np.abs(sigma).max() / R[k, h].min())


def _scale(tr, seed):
    rng = np.random.default_rng(seed)
    s = rng.choice([-1.0, 1.0], tr.n_nodes) / rng.uniform(5.0, 60.0, tr.n_nodes)
    s[rng.random(tr.n_nodes) < 0.3] = 0.0                 # unrated edges
    return s


def test_thermal_terms_are_the_path_minimum():
    zones, P = _cases()[0]
    for z_i, (tr, Pz) in enumerate(_each_zone(zones, P)):
        sc = _scale(tr, z_i)
        z = HR.zone_hosting(tr, Pz, UR, sc)
        th, _ = HR.thermal_terms(NR.zone_state(tr.parent, tr.r, tr.res_node, Pz)[0], sc)
        for h, v in enumerate(tr.res_node):
            path = []
            while v >= 0:
                path.append(v)
                v = tr.parent[v]
            assert np.array_equal(z["L"][tr.res_node[h]], th[path].min(axis=0))
        m = np.minimum(z["V"], z["L"])[tr.res_node]
        assert np.array_equal(z["cap"], np.where(m > 0.0, m, 0.0))


def test_uniform_matches_the_dense_row_sums():
    zones, P = _cases()[2]
    for tr, Pz in _each_zone(zones, P):
        res = np.asarray(tr.res_node, dtype=np.int64)
        R = tr.rmat()[np.ix_(res, res)]
        W = R.sum(axis=1)
        sigma = UR - R @ Pz
        k = W > 0.0
        ref = (sigma[k] / W[k, None]).min(axis=0)
        got = HR.zone_hosting(tr, Pz, UR)["uniform"]
        assert np.allclose(got, np.where(ref > 0.0, ref, 0.0), rtol=1e-12, atol=1e-15)


def test_uniform_thermal_term():
    """A single rated edge above every residence: the uniform headroom is its room over the residence count."""
    tr = FeederTree(parent=np.array([-1, 0, 1, 1], np.int32), r=np.array([1e-6, 1e-6, 1e-6, 1e-6]),
                    res_node=np.array([2, 3, 3], np.int32))
    P = np.array([[1.0, 2.0], [0.5, 0.0], [3.0, 1.0]])
    sc = np.array([1.0 / 20.0, 0.0, 0.0, 0.0])
    z = HR.zone_hosting(tr, P, UR, sc)
    F = P.sum(axis=0)
    assert np.array_equal(z["uniform"], (1.0 - sc[0] * F) / (sc[0] * 3.0))
    assert np.array_equal(z["cap"], np.broadcast_to((1.0 - sc[0] * F) / sc[0], (3, 2)))
    assert z["thermal"].all()


# Adding cap * (1 + 1e-6) raises the binding row by 1e-6 of its slack (the binding edge's loading by 1e-6 of its room).
# Rounding of D and of the loading stays below 1e-15, so the check is restricted to binding slacks (pu^2) and rooms
# (1 - |s| F) of at least 1e-6, where the added 1e-12 cannot be rounding.
BREAK_MIN = 1e-6


@pytest.mark.parametrize("case", range(3))
@pytest.mark.parametrize("rated", [False, True])
def test_adding_the_capacity_keeps_the_limits(case, rated):
    zones, P = _cases()[case]
    rng = np.random.default_rng(case)
    u = VHIGH * VHIGH - VSET * VSET
    checked = broke = 0
    for z_i, (tr, Pz) in enumerate(_each_zone(zones, P)):
        sc = _scale(tr, z_i) if rated else None
        z = HR.zone_hosting(tr, Pz, UR, sc)
        cand = np.argwhere((z["cap"] > 0.0) & np.isfinite(z["cap"]))
        if len(cand) == 0:
            continue
        res = np.asarray(tr.res_node, dtype=np.int64)
        cols = HR.RR._Columns(tr)
        for h, t in cand[rng.choice(len(cand), min(8, len(cand)), replace=False)]:
            cap = z["cap"][h, t]

            def state(add):
                Q = Pz.copy()
                Q[h, t] += add
                F, D = NR.zone_state(tr.parent, tr.r, tr.res_node, Q)
                load = np.zeros(len(F)) if sc is None else np.abs(sc * F[:, t])
                return D[res, t] - u, load

            c = cols(int(h))
            k = c > 0.0                                   # the rows and edges the home's load reaches (the others keep
            v, path = res[h], []                          # their bytes)
            while v >= 0:
                path.append(v)
                v = tr.parent[v]
            exc, load = state(cap)
            assert exc[k].max() <= TOL + 1e-15 and load[path].max() <= 1.0 + 1e-12
            checked += 1
            if z["V"][res[h], t] <= z["L"][res[h], t]:
                i = np.nonzero(k)[0][np.argmin(z["sigma"][res[k], t] / c[k])]
                slack = z["sigma"][res[i], t]
            else:
                _, room = HR.thermal_terms(NR.zone_state(tr.parent, tr.r, tr.res_node, Pz)[0][:, t:t + 1], sc)
                th = np.array([room[a, 0] / abs(sc[a]) if sc[a] != 0.0 else np.inf for a in path])
                slack = room[path[int(np.argmin(th))], 0]
            if slack >= BREAK_MIN:
                exc, load = state(cap * (1.0 + 1e-6))
                assert exc[k].max() > TOL or load[path].max() > 1.0
                broke += 1
    assert checked > 0 and broke > 0

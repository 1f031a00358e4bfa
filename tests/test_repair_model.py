"""CPU: the numpy model of the greedy voltage repair (tests/repair_ref.py) keeps every home's windows, never makes a row
worse, repairs what it reports as repaired (checked against the dense sensitivity matrix), and drops before it moves."""
import numpy as np
import pytest

import network_ref as NR
import repair_ref as RR
from revs_admm_b200.feeder import FeederTree, synthetic_feeder, synthetic_homes, synthetic_tariff


def _zones(seed):
    """Zones with several residences on one node and nodes without any, plus a one-node zone."""
    rng = np.random.default_rng(seed)
    out = []
    for n in (12, 30, 45):
        t = synthetic_feeder(n, seed=seed + n, laterals=2, r_secondary=3e-4)
        res = t.res_node.copy()
        res[1::4] = res[0]
        res[2::7] = rng.integers(0, t.n_nodes - n, len(res[2::7]))
        out.append(FeederTree(parent=t.parent, r=t.r, res_node=res.astype(np.int32)))
    out.insert(1, FeederTree(parent=np.array([-1], np.int32), r=np.array([1e-3]), res_node=np.zeros(4, np.int32)))
    return out


def _schedule(hm, T, rng):
    """A random binary schedule inside every home's windows: n_min <= count <= n_max hours of [start, end)."""
    H = len(hm["load"])
    nmin, nmax = RR.count_min(hm), RR.count_max(hm)
    bits = np.zeros((H, T), dtype=bool)
    for h in range(H):
        if not hm["has_ev"][h]:
            continue
        hours = np.arange(hm["start"][h], hm["end"][h])
        k = int(rng.integers(nmin[h], min(nmax[h], len(hours)) + 1))
        bits[h, rng.choice(hours, k, replace=False)] = True
    return hm["load"] + np.where(bits, hm["rating"][:, None], 0.0), bits


def _homes(H, T, seed):
    hm = synthetic_homes(H, T, seed=seed)
    rng = np.random.default_rng(seed)
    hm["initial"] = rng.uniform(0.05, 0.4, H)             # various SOC windows: some homes can drop hours
    sph = max(1, T // 24)
    hm["start"] = np.minimum(rng.integers(8, 13, H) * sph, T - 1).astype(np.int32)
    hm["end"] = np.minimum(hm["start"] + rng.integers(9, 14, H) * sph, T).astype(np.int32)
    k0 = np.maximum(1, ((hm["end"] - hm["start"]) * rng.uniform(0.2, 0.6, H)).astype(int))
    hm["capacity"] = hm["rating"] * (k0 - 0.05) / (0.9 - hm["initial"])     # n_min = k0 <= n_max
    return hm


def _case(T, seed, frac):
    zones = _zones(seed)
    H = sum(z.n_res for z in zones)
    hm = _homes(H, T, seed)
    rng = np.random.default_rng(seed + 1)
    P, bits = _schedule(hm, T, rng)
    cost = synthetic_tariff(T)
    drop = NR.network_check(zones, P)["drop"]
    u = frac * float(drop.max())                          # tight: the worst steps violate
    return zones, hm, P, bits, cost, u


def _excess(zones, P, u):
    out, off = [], 0
    for z in zones:
        _, D = NR.zone_state(z.parent, z.r, z.res_node, P[off:off + z.n_res])
        out.append(D[z.res_node] - u)
        off += z.n_res
    return out


@pytest.mark.parametrize("T", [24, 37, 96])
@pytest.mark.parametrize("frac", [0.6, 0.85])
def test_repair_properties(T, frac):
    row_tol = 1e-9
    zones, hm, P, bits, cost, u = _case(T, T, frac)
    out = RR.repair(zones, P, bits, hm, cost, vset=1.0, vhigh=np.sqrt(1.0 + u), row_tol=row_tol)
    u = np.sqrt(1.0 + u) ** 2 - 1.0                       # the model's u, rounded as it rounds it
    info, B, Pr = out["zone_info"], out["bits"], out["P_sch"]
    nmin, nmax = RR.count_min(hm), RR.count_max(hm)
    t = np.arange(T)[None, :]
    inwin = (t >= hm["start"][:, None]) & (t < hm["end"][:, None])
    ev = hm["has_ev"] > 0
    cnt = B.sum(axis=1)
    assert not B[~ev].any() and not (B & ~inwin).any()
    assert (cnt[ev] >= nmin[ev]).all() and (cnt[ev] <= nmax[ev]).all()
    assert np.array_equal(Pr, hm["load"] + np.where(B, hm["rating"][:, None], 0.0))
    assert (info[:, 0] > 0).any() and info[:, 1:].sum() > 0
    ex0, ex1 = _excess(zones, P, u), _excess(zones, Pr, u)
    off = 0
    for z, (st, mv, dr), e0, e1 in zip(zones, info, ex0, ex1):
        s = slice(off, off + z.n_res)
        off += z.n_res
        if st == 0:
            assert np.array_equal(Pr[s], P[s]) and mv == 0 and dr == 0
            continue
        assert (e1 <= np.maximum(e0, row_tol)).all()
        feasible = (e0 <= row_tol).all(axis=0)
        assert (e1[:, feasible] <= row_tol).all()
        violated = (e0 > row_tol).any(axis=0)
        assert mv + dr <= int(bits[s][:, violated].sum())
        if st == 1:
            Rres = z.rmat()[np.ix_(z.res_node, z.res_node)]
            assert ((Rres @ Pr[s]) - u <= row_tol + 1e-12).all()
        else:
            assert (e1 > row_tol).any()
    # homes whose hours did not change keep their bytes
    same = (B == bits).all(axis=1)
    assert np.array_equal(Pr[same], P[same])


def test_base_load_violation_is_left():
    T = 24
    zones, hm, P, bits, cost, _ = _case(T, 3, 0.8)
    base = NR.network_check(zones, hm["load"])["drop"].max()
    u = 0.9 * float(base)
    vhigh = np.sqrt(1.0 + u)
    out = RR.repair(zones, P, bits, hm, cost, vset=1.0, vhigh=vhigh, row_tol=1e-9)
    assert (out["zone_info"][:, 0] == 2).any()
    nmin = RR.count_min(hm)
    ev = hm["has_ev"] > 0
    assert (out["bits"].sum(axis=1)[ev] >= nmin[ev]).all()


def test_a_home_above_n_min_drops():
    """One node, one charging home with a spare hour: the worst step's hour is dropped, not moved."""
    T = 24
    z = FeederTree(parent=np.array([-1], np.int32), r=np.array([1e-3]), res_node=np.zeros(2, np.int32))
    hm = dict(load=np.full((2, T), 0.5), has_ev=np.array([1, 0], np.uint8), rating=np.array([4.8, 0.0]),
              capacity=np.array([20.0, 1.0]), initial=np.array([0.2, 0.0]), start=np.array([6, 0], np.int32),
              end=np.array([20, 0], np.int32))
    hm["load"][:, 10] = 0.9                                # step 10 is the worst
    nmin = int(RR.count_min(hm)[0])
    bits = np.zeros((2, T), dtype=bool)
    bits[0, 8:8 + nmin + 1] = True                         # one hour above n_min, including step 10
    P = hm["load"] + np.where(bits, hm["rating"][:, None], 0.0)
    u = 2e-3 * (4.8 + 1.0) - 1e-4                          # every charging step violates; with the charger off none does
    out = RR.repair([z], P, bits, hm, synthetic_tariff(T), vset=1.0, vhigh=np.sqrt(1.0 + u), row_tol=1e-9)
    st, mv, dr = out["zone_info"][0]
    assert dr == 1 and not out["bits"][0, 10] and out["bits"][0].sum() == nmin

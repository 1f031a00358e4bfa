"""CPU checks of the population network check: the numpy model of tests/network_ref.py against the dense sensitivity
matrix and against a brute-force reduction, and PipelinedSolver's merge of per-pipeline summaries."""
import itertools

import numpy as np

import network_ref as NR
import revs_oracle as O
from revs_admm_b200.feeder import FeederTree, reference_shaped_feeder, split_zones, synthetic_feeder
from revs_admm_b200.parallel import merge_network_summaries


def _zones(seed):
    """Small zones with several residences on one node, nodes without residences, a one-node zone and a zone with
    two roots."""
    rng = np.random.default_rng(seed)
    out = []
    for n in (9, 23):
        t = synthetic_feeder(n, seed=seed + n, laterals=2)
        res = t.res_node.copy()
        res[1::3] = res[0]                                          # three residences on the first residence's node
        res[2] = int(rng.integers(0, t.n_nodes - n))                # one on a transformer node
        out.append(FeederTree(parent=t.parent, r=t.r, res_node=res.astype(np.int32)))
    out.append(FeederTree(parent=np.array([-1], np.int32), r=np.array([2e-3]), res_node=np.zeros(3, np.int32)))
    out.append(FeederTree(parent=np.array([-1, 0, -1, 2, 1], np.int32), r=rng.uniform(1e-4, 1e-3, 5),
                          res_node=np.array([4, 3, 1, 4], np.int32)))
    return out


def _subtree_sums(tr, P):
    """Flow on the edge above every node: sum of the schedules of the residences below it (path indicators)."""
    F = np.zeros((tr.n_nodes, P.shape[1]))
    for j, v in enumerate(tr.res_node):
        while v >= 0:
            F[v] += P[j]
            v = tr.parent[v]
    return F


def test_model_matches_dense_sensitivity_and_subtree_sums():
    for seed, T in ((0, 24), (1, 37), (2, 5)):
        rng = np.random.default_rng(seed)
        for tr in _zones(seed):
            P = rng.uniform(-1.0, 6.0, (tr.n_res, T))
            F, D = NR.zone_state(tr.parent, tr.r, tr.res_node, P)
            Pall = np.zeros((tr.n_nodes, T))
            np.add.at(Pall, tr.res_node, P)
            R = O.rmat_from_tree(tr.parent, tr.r)
            assert np.abs(D - R @ Pall).max() <= 1e-12 * max(1.0, np.abs(D).max())
            assert np.abs(F - _subtree_sums(tr, P)).max() <= 1e-12 * np.abs(F).max()
            assert np.abs(D[tr.res_node] - tr.drop(P)).max() <= 1e-12 * max(1.0, np.abs(D).max())


def test_model_on_reference_shaped_zones():
    T = 96
    zones = [z for z, _ in split_zones(reference_shaped_feeder(600, seed=4, r_scale=0.7))]
    rng = np.random.default_rng(3)
    for tr in zones:
        P = rng.uniform(0.0, 8.0, (tr.n_res, T))
        F, D = NR.zone_state(tr.parent, tr.r, tr.res_node, P)
        Pall = np.zeros((tr.n_nodes, T))
        np.add.at(Pall, tr.res_node, P)
        assert np.abs(D - O.rmat_from_tree(tr.parent, tr.r) @ Pall).max() <= 1e-12 * np.abs(D).max()
        assert np.abs(D[tr.res_node] - tr.drop(P)).max() <= 1e-12 * np.abs(D).max()


def _brute_summary(zones, P, vset, vlow, vhigh, row_tol, scale):
    """The summary by enumeration of every (zone, index, step) in order: the first strictly larger value wins."""
    v2 = vset * vset
    u, low = vhigh * vhigh - v2, v2 - vlow * vlow
    best = {k: (-np.inf, -1, -1, -1) for k in ("drop", "exc", "load")}
    rows = nlow = over = 0
    off = noff = 0
    for z, tr in enumerate(zones):
        F, D = NR.zone_state(tr.parent, tr.r, tr.res_node, P[off:off + tr.n_res])
        L = F if scale is None else scale[noff:noff + tr.n_nodes, None] * F
        T = D.shape[1]
        for i, t in itertools.product(range(tr.n_nodes), range(T)):
            if D[i, t] > best["drop"][0]:
                best["drop"] = (D[i, t], z, i, t)
            if abs(L[i, t]) > best["load"][0]:
                best["load"] = (abs(L[i, t]), z, i, t)
            nlow += D[i, t] > low
            over += scale is not None and abs(L[i, t]) > 1.0
        for j, t in itertools.product(range(tr.n_res), range(T)):
            e = D[tr.res_node[j], t] - u
            if e > best["exc"][0]:
                best["exc"] = (e, z, j, t)
            rows += e > row_tol
        off += tr.n_res
        noff += tr.n_nodes
    return best, rows, nlow, over


def test_summary_tie_rule_and_counts():
    T = 6
    base = _zones(5)
    zones = [base[0], base[0], base[2], base[3], base[1]]           # zone 1 repeats zone 0: exact ties across zones
    rng = np.random.default_rng(7)
    P0 = rng.uniform(0.0, 5.0, (base[0].n_res, T))
    P0[:, 2] = P0[:, 1]                                             # steps 1 and 2 tie
    P0[0, :] = 0.0
    P = np.concatenate([P0, P0] + [rng.uniform(0.0, 0.05, (z.n_res, T)) for z in zones[2:]])    # zones 0 and 1 lead
    P[-zones[-1].n_res:] = 0.0                                      # a zone without load: every value ties at 0
    n_all = sum(z.n_nodes for z in zones)
    scale = rng.choice([-1.0, 1.0], n_all) / rng.uniform(5.0, 60.0, n_all)
    for sc in (None, scale):
        kw = dict(vset=1.03, vlow=0.95, vhigh=1.05, row_tol=1e-9)
        got = NR.network_check(zones, P, scale=sc, **kw)
        best, rows, nlow, over = _brute_summary(zones, P, scale=sc, **kw)
        s = got["summary"]
        assert (s["drop_max"], s["drop_zone"], s["drop_node"], s["drop_step"]) == best["drop"]
        assert (s["row_excess_max"], s["excess_zone"], s["excess_res"], s["excess_step"]) == best["exc"]
        assert (s["loading_max"], s["loading_zone"], s["loading_node"], s["loading_step"]) == best["load"]
        assert (s["rows_violated"], s["nodes_below_vlow"], s["edges_overloaded"]) == (rows, nlow, over)
        assert s["drop_zone"] == 0 and s["v_min"] == np.sqrt(1.03 * 1.03 - s["drop_max"])
        assert np.array_equal(got["zone_worst"][0, :2], got["zone_worst"][1, :2])


def test_merge_of_pipeline_summaries():
    T = 8
    base = _zones(11)
    zones = [base[1], base[0], base[1], base[3], base[2], base[0]]
    rng = np.random.default_rng(2)
    P = np.concatenate([rng.uniform(0.0, 5.0, (z.n_res, T)) for z in zones])
    P[base[1].n_res + base[0].n_res:][:base[1].n_res] = P[:base[1].n_res]     # zone 2 == zone 0: the maxima tie
    n_all = sum(z.n_nodes for z in zones)
    scale = rng.uniform(-0.1, 0.1, n_all)
    whole = NR.network_check(zones, P, scale=scale, vset=1.0, vlow=0.97, vhigh=1.02)["summary"]
    for cuts in ([(0, 2), (2, 6)], [(0, 1), (1, 3), (3, 4), (4, 6)], [(0, 6)]):
        parts = []
        for a, b in cuts:
            h0, h1 = sum(z.n_res for z in zones[:a]), sum(z.n_res for z in zones[:b])
            n0, n1 = sum(z.n_nodes for z in zones[:a]), sum(z.n_nodes for z in zones[:b])
            parts.append(NR.network_check(zones[a:b], P[h0:h1], scale=scale[n0:n1], vset=1.0, vlow=0.97,
                                          vhigh=1.02)["summary"])
        assert merge_network_summaries(parts, [a for a, _ in cuts]) == whole


def test_merge_skips_parts_without_candidates():
    none = dict(drop_max=0.5, v_min=0.7, drop_zone=0, drop_node=3, drop_step=1, row_excess_max=-np.inf, excess_zone=-1,
                excess_res=-1, excess_step=-1, rows_violated=0, nodes_below_vlow=4, loading_max=2.0, loading_zone=0,
                loading_node=1, loading_step=0, edges_overloaded=5)
    some = dict(none, drop_max=0.5, v_min=0.7, drop_zone=1, drop_node=0, drop_step=0, row_excess_max=-0.25,
                excess_zone=0, excess_res=2, excess_step=3, rows_violated=1, nodes_below_vlow=1, loading_max=2.0,
                loading_zone=0, loading_node=0, loading_step=0, edges_overloaded=2)
    m = merge_network_summaries([none, some], [0, 4])
    assert (m["drop_zone"], m["drop_node"], m["drop_step"]) == (0, 3, 1)            # tie on value: lower zone
    assert (m["row_excess_max"], m["excess_zone"], m["excess_res"], m["excess_step"]) == (-0.25, 4, 2, 3)
    assert (m["loading_zone"], m["loading_node"]) == (0, 1)
    assert (m["rows_violated"], m["nodes_below_vlow"], m["edges_overloaded"]) == (1, 5, 7)
    m = merge_network_summaries([none, none], [0, 1])
    assert m["row_excess_max"] == -np.inf and m["excess_zone"] == -1

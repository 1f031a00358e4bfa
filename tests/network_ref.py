"""numpy model of the population network check (csrc/network_check.cu, include/revs_admm.h: revs_network_check).

The recurrences of FeederTree.drop extended to the line flows and to the summary:
    F_i = inj_i + sum_{children c} F_c      leaves -> root   (flow on the edge above node i)
    D_i = D_parent(i) + 2 r_i F_i           root -> leaves   (D = R P at node i)
with r_i = cumr[i] - cumr[parent[i]] and the sums in the kernel's order (a node's residences by home index, then its
children by node index), so that voltage and loading equal the device's bit for bit."""
import numpy as np


def zone_state(parent, r, res_node, P):
    """F and D of one zone, both [n_nodes, T], for the schedule P [n_res, T] of its residences."""
    parent = np.asarray(parent, dtype=np.int64)
    res_node = np.asarray(res_node, dtype=np.int64)
    n = len(parent)
    P = np.asarray(P, dtype=np.float64).reshape(len(res_node), -1)
    T = P.shape[1]
    c = np.zeros(n)
    for i in range(n):                      # the library's cumulative resistances (revs_set_feeder_tree(s))
        c[i] = (c[parent[i]] if parent[i] >= 0 else 0.0) + r[i]
    rr = np.where(parent >= 0, c - c[np.maximum(parent, 0)], c)
    F = np.zeros((n, T))
    for j in range(len(res_node)):
        F[res_node[j]] += P[j]
    children = [[] for _ in range(n)]
    for i in range(n):
        if parent[i] >= 0:
            children[parent[i]].append(i)
    for i in range(n - 1, -1, -1):
        for ch in children[i]:
            F[i] += F[ch]
    D = np.empty((n, T))
    for i in range(n):
        D[i] = (D[parent[i]] if parent[i] >= 0 else 0.0) + (2.0 * rr[i]) * F[i]
    return F, D


def _first_max(a):
    """(max, flat index of its first occurrence) of a 2-D array; (-inf, -1) when empty."""
    if a.size == 0:
        return -np.inf, -1
    k = int(np.argmax(a))
    return float(a.flat[k]), k


def summarize(zones, D, L, vset, vlow, vhigh, row_tol, scaled):
    """Summary and zone_worst from the drops D and loadings L of every zone (lists of [n_nodes, T] arrays): maxima
    to the largest value, ties to the lowest (zone, index, step), integer counts."""
    v2 = vset * vset
    u, low = vhigh * vhigh - v2, v2 - vlow * vlow
    s = dict(drop_max=-np.inf, v_min=np.nan, drop_zone=-1, drop_node=-1, drop_step=-1,
             row_excess_max=-np.inf, excess_zone=-1, excess_res=-1, excess_step=-1,
             rows_violated=0, nodes_below_vlow=0,
             loading_max=-np.inf, loading_zone=-1, loading_node=-1, loading_step=-1, edges_overloaded=0)
    zw = np.empty((len(zones), 3))
    for z, (tr, Dz, Lz) in enumerate(zip(zones, D, L)):
        T = Dz.shape[1]
        E = Dz[np.asarray(tr.res_node, dtype=np.int64)] - u
        A = np.abs(Lz)
        for arr, val, zk, ik, tk, col in ((Dz, "drop_max", "drop_zone", "drop_node", "drop_step", 0),
                                          (E, "row_excess_max", "excess_zone", "excess_res", "excess_step", 1),
                                          (A, "loading_max", "loading_zone", "loading_node", "loading_step", 2)):
            m, k = _first_max(arr)
            zw[z, col] = m
            if k >= 0 and m > s[val]:       # strict: an equal value of a later zone loses
                s.update({val: m, zk: z, ik: k // T, tk: k % T})
        s["rows_violated"] += int((E > row_tol).sum())
        s["nodes_below_vlow"] += int((Dz > low).sum())
        if scaled:
            s["edges_overloaded"] += int((A > 1.0).sum())
    s["v_min"] = float(np.sqrt(v2 - s["drop_max"]))
    return s, zw


def network_check(zones, P, vset=1.0, vlow=0.95, vhigh=1.05, row_tol=1e-9, scale=None):
    """What Solver.network_check(P, ..., full=True, zones=True) returns, plus the drops D [total nodes, T].
    zones: FeederTree-like (parent, r, res_node) in solver order, P [H, T] in that home order, scale [total nodes]."""
    P = np.asarray(P, dtype=np.float64)
    D, L, off, noff = [], [], 0, 0
    for tr in zones:
        F, Dz = zone_state(tr.parent, tr.r, tr.res_node, P[off:off + len(tr.res_node)])
        n = len(tr.parent)
        L.append(F if scale is None else np.asarray(scale, dtype=np.float64)[noff:noff + n, None] * F)
        D.append(Dz)
        off += len(tr.res_node)
        noff += n
    summary, zw = summarize(zones, D, L, vset, vlow, vhigh, row_tol, scale is not None)
    Dall = np.concatenate(D)
    return dict(summary=summary, voltage=np.sqrt(vset * vset - Dall), loading=np.concatenate(L), zone_worst=zw,
                drop=Dall)

"""numpy model of the greedy voltage repair (csrc/repair.cu, include/revs_admm.h: revs_repair_schedule).

The exact rule and operation order of the kernel: initial drops D = R P at the residences in the network check's
order (network_ref.zone_state), R[i,h] = 2 cumr[lca(node i, node h)], every value rounded as the kernel rounds it
(D - a, D + a, (D + a) - u, D - u, rating * R), maxima under the same total orders.  So the device result equals
this model bit for bit."""
import numpy as np

import network_ref as NR


def count_min(hm):
    """n_min of every home: the SOC target as a count of charging hours (revs_capi.cu count_window)."""
    step = np.asarray(hm["rating"], dtype=np.float64) / np.asarray(hm["capacity"], dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):     # homes without EV (rating 0) never charge
        lo = np.ceil((0.9 - np.asarray(hm["initial"], dtype=np.float64)) / step - 1e-9)
    return np.where(np.isfinite(lo), np.maximum(lo, 0), 0).astype(np.int64)


def count_max(hm):
    step = np.asarray(hm["rating"], dtype=np.float64) / np.asarray(hm["capacity"], dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        hi = np.floor((1.0 - np.asarray(hm["initial"], dtype=np.float64)) / step + 1e-9)
    return np.where(np.isfinite(hi), hi, 0).astype(np.int64)


class _Columns:
    """R[:, h] of one zone's residences from the tree (2 cumr at the lowest common ancestor), cached per home."""

    def __init__(self, tr):
        parent = np.asarray(tr.parent, dtype=np.int64)
        n = len(parent)
        c, depth = np.zeros(n), np.zeros(n, dtype=np.int64)
        for i in range(n):
            c[i] = (c[parent[i]] if parent[i] >= 0 else 0.0) + tr.r[i]
            depth[i] = depth[parent[i]] + 1 if parent[i] >= 0 else 0
        self.parent, self.c, self.res = parent, c, np.asarray(tr.res_node, dtype=np.int64)
        self.levels = [np.nonzero(depth == d)[0] for d in range(int(depth.max()) + 1 if n else 0)]
        self.cache = {}

    def __call__(self, h):
        if h not in self.cache:
            on = np.zeros(len(self.parent), dtype=bool)
            q = int(self.res[h])
            while q >= 0:
                on[q] = True
                q = int(self.parent[q])
            val = np.zeros(len(self.parent))          # 2 cumr of the deepest node of h's root path above every node
            for lv in self.levels:
                up = np.where(self.parent[lv] >= 0, val[np.maximum(self.parent[lv], 0)], 0.0)
                val[lv] = np.where(on[lv], 2.0 * self.c[lv], up)
            self.cache[h] = val[self.res]
        return self.cache[h]


def repair_zone(tr, P, bits, load, rating, start, end, nmin, cost, u, row_tol):
    """One zone: P [n, T] its schedule, bits [n, T] its charging decisions.  Returns (P, bits, (status, moves, drops),
    D [n, T] drops of the result)."""
    n, T = P.shape
    P, bits = P.copy(), bits.copy()
    _, Dn = NR.zone_state(tr.parent, tr.r, tr.res_node, P)
    D = Dn[np.asarray(tr.res_node, dtype=np.int64)].copy()
    if n == 0 or not ((D - u).max() > row_tol):
        return P, bits, (0, 0, 0), D
    R = _Columns(tr)
    order = sorted(range(T), key=lambda t: (cost[t], t))
    wv, wi = np.empty(T), np.empty(T, dtype=np.int64)

    def worst(t):
        x = D[:, t] - u
        i = int(np.argmax(x))
        wv[t], wi[t] = x[i], i

    for t in range(T):
        worst(t)
    count = bits.sum(axis=1)
    stuck = np.zeros(T, dtype=bool)
    moves = drops = 0
    while True:
        steps = [t for t in range(T) if not stuck[t] and wv[t] > row_tol]
        if not steps:
            break
        ts = min(steps, key=lambda t: (-wv[t], wi[t], t))
        i_s = int(wi[ts])
        homes = np.nonzero(bits[:, ts])[0]
        rel = {int(h): rating[h] * R(int(h))[i_s] for h in homes}
        done = False
        for h in sorted(rel, key=lambda h: (-rel[h], h)):
            a = rating[h] * R(h)
            tp = -1
            if count[h] <= nmin[h]:
                tp = None
                for t in order:
                    if t < start[h] or t >= end[h] or bits[h, t]:
                        continue
                    if not ((D[:, t] + a) - u > row_tol).any():
                        tp = t
                        break
                if tp is None:
                    continue
            D[:, ts] = D[:, ts] - a
            bits[h, ts] = False
            P[h, ts] = load[h, ts] + 0.0
            if tp >= 0:
                D[:, tp] = D[:, tp] + a
                bits[h, tp] = True
                P[h, tp] = load[h, tp] + rating[h]
                moves += 1
            else:
                count[h] -= 1
                drops += 1
            worst(ts)
            if tp >= 0:
                worst(tp)
            done = True
            break
        if not done:
            stuck[ts] = True
    return P, bits, (2 if stuck.any() else 1, moves, drops), D


def repair(zones, P, bits, hm, cost, vset=1.0, vhigh=1.05, row_tol=1e-9):
    """What Solver.repair_schedule returns, for the schedule P [H, T] and its charging decisions bits [H, T] (bool) of
    the zones (FeederTree-like, solver order): dict(P_sch, bits, zone_info [zones, 3])."""
    u = vhigh * vhigh - vset * vset
    P, bits = np.asarray(P, dtype=np.float64), np.asarray(bits, dtype=bool)
    nmin = count_min(hm)
    outP, outB, info, off = P.copy(), bits.copy(), [], 0
    for tr in zones:
        s = slice(off, off + tr.n_res)
        outP[s], outB[s], zi, _ = repair_zone(tr, P[s], bits[s], hm["load"][s], hm["rating"][s], hm["start"][s],
                                              hm["end"][s], nmin[s], np.asarray(cost, dtype=np.float64), u, row_tol)
        info.append(zi)
        off += tr.n_res
    return dict(P_sch=outP, bits=outB, zone_info=np.array(info, dtype=np.int32).reshape(-1, 3))


def unpack(mask, T):
    """[H, T] bool from the [H, ceil(T/64)] uint64 hour masks."""
    mask = np.asarray(mask, dtype=np.uint64)
    t = np.arange(T)
    return ((mask[:, t // 64] >> (t % 64).astype(np.uint64)) & np.uint64(1)).astype(bool)

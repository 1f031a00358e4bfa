"""numpy model of the bracket of the centralized optimum (csrc/central.cu, include/revs_admm.h: revs_central_bracket).

The kernels' rule and operation order: R x at the residences in the network check's order (network_ref.zone_state),
the greedy repair of repair_ref.repair_zone, every value rounded as the kernels round it, and every per-zone sum in
their fixed order (fsum).  So the device result equals this model bit for bit."""
import numpy as np

import network_ref as NR
import repair_ref as RR

THREADS, WARPS, STALL = 256, 8, 20


def fsum(x):
    """Sum of a zone's [n, T] array in the kernels' order: thread k adds the elements k, k + 256, ... of the flattened
    array, a warp butterfly adds the threads of a warp, thread 0 adds the warps in order."""
    v = np.asarray(x, dtype=np.float64).ravel()
    rows = np.concatenate([v, np.zeros((-v.size) % THREADS)]).reshape(-1, THREADS)
    lane = np.cumsum(np.vstack([np.zeros(THREADS), rows]), axis=0)[-1]      # 0.0 + x0 + x1 + ..., one add at a time
    idx = np.arange(THREADS)
    for o in (16, 8, 4, 2, 1):
        lane = lane + lane[idx ^ o]
    s = lane[0]
    for w in range(1, WARPS):
        s = s + lane[32 * w]
    return float(s)


def select(r, nmin, nmax):
    """Priced selection from the reduced costs r [n, T] (+inf outside the window): the n_min smallest, then further
    hours while negative, up to n_max; ties to the earliest hour."""
    n, T = r.shape
    order = np.argsort(r, axis=1, kind="stable")
    rank = np.empty_like(order)
    np.put_along_axis(rank, order, np.broadcast_to(np.arange(T), (n, T)).copy(), axis=1)
    return (r < np.inf) & ((rank < nmin[:, None]) | ((rank < nmax[:, None]) & (r < 0.0)))


class _Zone:
    def __init__(self, tr, hz, cost):
        self.tr, self.cost = tr, np.asarray(cost, dtype=np.float64)
        self.res = np.asarray(tr.res_node, dtype=np.int64)
        self.load = np.asarray(hz["load"], dtype=np.float64)
        self.rating = np.asarray(hz["rating"], dtype=np.float64)
        self.start, self.end = np.asarray(hz["start"]), np.asarray(hz["end"])
        ev = np.asarray(hz["has_ev"]) > 0
        T = self.load.shape[1]
        t = np.arange(T)[None, :]
        self.win = ev[:, None] & (t >= self.start[:, None]) & (t < self.end[:, None])
        self.nmin = np.where(ev, RR.count_min(hz), 0)
        self.nmax = np.where(ev, RR.count_max(hz), 0)
        if (ev & ((self.nmin > self.nmax) | (self.nmin > self.win.sum(axis=1)))).any():
            raise ValueError("a home's SOC target needs more hours than its plug-in window has")

    def R(self, x):
        return NR.zone_state(self.tr.parent, self.tr.r, self.tr.res_node, x)[1][self.res]

    def P(self, e):
        return self.load + np.where(e, self.rating[:, None], 0.0)

    def priced(self, y):
        red = self.rating[:, None] * (self.cost[None, :] + self.R(y))
        return select(np.where(self.win, red, np.inf), self.nmin, self.nmax)

    def repair(self, e, u, row_tol):
        P, bits, info, _ = RR.repair_zone(self.tr, self.P(e), e, self.load, self.rating, self.start, self.end,
                                          self.nmin, self.cost, u, row_tol)
        c = fsum(self.cost[None, :] * P)
        return P, bits, info, np.inf if info[0] == 2 else c


def bracket_zone(tr, hz, cost, u, row_tol, iters):
    """One zone: (P [n, T] kept schedule, bits [n, T], (LB, UB), (status, ascent steps, moves + drops))."""
    Z = _Zone(tr, hz, cost)
    c = Z.cost[None, :]
    n, T = Z.load.shape
    emax = select(np.where(Z.win, -(Z.rating[:, None] * c), np.inf), Z.nmin, Z.nmax)
    cmax = fsum(c * Z.P(emax))
    y = np.zeros((n, T))
    e = Z.priced(y)
    P = Z.P(e)
    P1, b1, i1, ub = Z.repair(e, u, row_tol)
    D = Z.R(P)
    yb, lb, theta, stall, steps, k = y, -np.inf, 1.0, 0, 0, 0
    while True:
        G = D - u
        g = np.where(y > 0.0, G, np.where(G > 0.0, G, 0.0))
        phi = fsum(c * P) + fsum(y * G)
        g2 = fsum(g * g)
        if phi > lb:
            lb, stall, yb = phi, 0, y
        else:
            stall += 1
            if stall == STALL:
                theta, stall = theta * 0.5, 0
        known = ub < np.inf
        if k >= iters or not g2 > 0.0 or ((ub - lb) <= 1e-9 * abs(ub) if known else lb > cmax):
            break
        target = ub if known else cmax + 0.01 * abs(cmax)
        alpha = theta * (target - phi) / g2
        steps += 1
        v = y + alpha * G
        y = np.where(v > 0.0, v, 0.0)
        k += 1
        P = Z.P(Z.priced(y))
        D = Z.R(P)
    P2, b2, i2, ub2 = Z.repair(Z.priced(yb), u, row_tol)
    first = i1[0]
    if ub2 < ub:
        P1, b1, i1, ub = P2, b2, i2, ub2
    status = 0 if first == 0 else 1 if ub < np.inf else 3 if lb > cmax else 2
    return P1, b1, (lb, ub), (status, steps, int(i1[1] + i1[2]))


def bracket(zones, hm, cost, vset=1.0, vhigh=1.05, row_tol=1e-9, iters=100):
    """What Solver.central_bracket returns for the zones (FeederTree-like, solver order) and homes hm:
    dict(P_sch [H, T], bits [H, T], zone_bounds [zones, 2], zone_info [zones, 3] int32)."""
    u = vhigh * vhigh - vset * vset
    H, T = np.asarray(hm["load"]).shape
    P, bits = np.empty((H, T)), np.zeros((H, T), dtype=bool)
    bounds, info, off = [], [], 0
    for tr in zones:
        s = slice(off, off + tr.n_res)
        hz = {k: np.asarray(v)[s] for k, v in hm.items()}
        P[s], bits[s], b, i = bracket_zone(tr, hz, cost, u, row_tol, iters)
        bounds.append(b)
        info.append(i)
        off += tr.n_res
    return dict(P_sch=P, bits=bits, zone_bounds=np.array(bounds, dtype=np.float64).reshape(-1, 2),
                zone_info=np.array(info, dtype=np.int32).reshape(-1, 3))

"""numpy model of the hosting capacity (csrc/hosting.cu, include/revs_admm.h: revs_hosting_capacity).

F and D come from network_ref.zone_state (the network check's recurrences and order), then the kernel's two further
passes in its arithmetic: sigma = (u + row_tol) - D at the residence nodes, M = the smallest sigma below every node,
V = the running minimum of M / (2 cumr) from the root down, L = the running minimum of the rated edges' thermal terms
(1 - |s| F) / |s|.  Every value is rounded as the kernel rounds it and every further step is a minimum, so the device
result equals this model bit for bit.  `brute_voltage` is the definition min_i sigma_i / R[i,h] over R[i,h] > 0."""
import numpy as np

import network_ref as NR
import repair_ref as RR


def _cumr(parent, r):
    c = np.zeros(len(parent))
    for i in range(len(parent)):
        c[i] = (c[parent[i]] if parent[i] >= 0 else 0.0) + r[i]
    return c


def thermal_terms(F, scale):
    """(1 - |s| F) / |s| of every rated edge, +inf on the unrated ones (s = 0 or scale None); also 1 - |s| F."""
    if scale is None:
        return np.full(F.shape, np.inf), None
    s = np.abs(np.asarray(scale, dtype=np.float64))[:, None]
    room = 1.0 - s * F
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(s != 0.0, room / s, np.inf), room


def zone_hosting(tr, P, ur, scale=None):
    """One zone, P [n_res, T], ur = u + row_tol, scale [n_nodes] or None: dict(cap [n_res, T], uniform [T],
    V, L [n_nodes, T] (the running minima at every node), sigma [n_nodes, T])."""
    parent = np.asarray(tr.parent, dtype=np.int64)
    res = np.asarray(tr.res_node, dtype=np.int64)
    n = len(parent)
    P = np.asarray(P, dtype=np.float64).reshape(len(res), -1)
    T = P.shape[1]
    F, D = NR.zone_state(tr.parent, tr.r, tr.res_node, P)
    N, W = NR.zone_state(tr.parent, tr.r, tr.res_node, np.ones((len(res), 1)))
    has = np.zeros(n, dtype=bool)
    has[res] = True
    sigma = ur - D
    th, room = thermal_terms(F, scale)
    um = np.full(T, np.inf)
    with np.errstate(divide="ignore", invalid="ignore"):
        rw = has & (W[:, 0] > 0.0)
        if rw.any():
            um = np.minimum(um, (sigma[rw] / W[rw]).min(axis=0))
        if scale is not None:
            s = np.abs(np.asarray(scale, dtype=np.float64))
            re = (s != 0.0) & (N[:, 0] > 0.0)
            if re.any():
                um = np.minimum(um, (room[re] / (s[re] * N[re, 0])[:, None]).min(axis=0))
    M = np.where(has[:, None], sigma, np.inf)
    for i in range(n - 1, -1, -1):                    # parent[i] < i: every child before its parent
        if parent[i] >= 0:
            M[parent[i]] = np.minimum(M[parent[i]], M[i])
    d = 2.0 * _cumr(parent, tr.r)
    V, L = np.empty((n, T)), th.copy()
    for i in range(n):
        with np.errstate(divide="ignore", invalid="ignore"):
            V[i] = M[i] / d[i] if d[i] > 0.0 else np.inf
        if parent[i] >= 0:
            V[i] = np.minimum(V[i], V[parent[i]])
            L[i] = np.minimum(L[i], L[parent[i]])
    m = np.minimum(V, L)[res]
    return dict(cap=np.where(m > 0.0, m, 0.0), uniform=np.where(um > 0.0, um, 0.0), V=V, L=L, sigma=sigma,
                thermal=(L < V)[res])


def hosting(zones, P, vset=1.0, vhigh=1.05, row_tol=1e-9, scale=None, hm=None):
    """What Solver.hosting_capacity(P, ...) returns for the zones (FeederTree-like, solver order), P [H, T] and the
    homes hm (None: the counts of window steps are 0, as before set_homes): dict(home_cap, zone_uniform, zone_counts)."""
    P = np.asarray(P, dtype=np.float64)
    H, T = P.shape
    ur = (vhigh * vhigh - vset * vset) + row_tol
    cap, uni, cnt = np.empty((H, T)), [], []
    off = noff = 0
    t = np.arange(T)[None, :]
    for tr in zones:
        hs = slice(off, off + tr.n_res)
        sc = None if scale is None else np.asarray(scale, dtype=np.float64)[noff:noff + tr.n_nodes]
        z = zone_hosting(tr, P[hs], ur, sc)
        cap[hs] = z["cap"]
        uni.append(z["uniform"])
        if hm is None:
            win = np.zeros((tr.n_res, T), dtype=bool)
            rating = np.zeros(tr.n_res)
        else:
            ev = np.asarray(hm["has_ev"])[hs] > 0
            win = ev[:, None] & (t >= np.asarray(hm["start"])[hs, None]) & (t < np.asarray(hm["end"])[hs, None])
            rating = np.asarray(hm["rating"], dtype=np.float64)[hs]
        cnt.append([int(win.sum()), int((win & (z["cap"] >= rating[:, None])).sum()), int(z["thermal"].sum())])
        off += tr.n_res
        noff += tr.n_nodes
    return dict(home_cap=cap, zone_uniform=np.array(uni).reshape(len(zones), T),
                zone_counts=np.array(cnt, dtype=np.int64).reshape(len(zones), 3))


def brute_voltage(tr, P, ur):
    """max(0, min_i sigma_i / R[i,h]) over the residences i with R[i,h] > 0, R[i,h] = 2 cumr[lca] (repair_ref._Columns),
    for every residence h of one zone: [n_res, T], +inf where no R[i,h] is positive."""
    res = np.asarray(tr.res_node, dtype=np.int64)
    D = NR.zone_state(tr.parent, tr.r, tr.res_node, P)[1][res]
    sigma = ur - D
    cols = RR._Columns(tr)
    out = np.full(D.shape, np.inf)
    for h in range(len(res)):
        c = cols(h)
        k = c > 0.0
        if k.any():
            out[h] = (sigma[k] / c[k, None]).min(axis=0)
    return np.where(out > 0.0, out, 0.0)

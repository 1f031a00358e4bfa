"""numpy model of the certificate of voltage infeasibility (csrc/certify.cu, include/revs_admm.h:
revs_certify_infeasible).

The kernels' rule and operation order: D0 = R load at the residences in the network check's order
(network_ref.zone_state), a_h(i) = rating_h R[i,h] with R[i,h] = 2 cumr[lca] (repair_ref._Columns), every fit test
(D0 + s) - u <= row_tol + 1e-12 with s summed one coefficient at a time in ascending order, maxima under the same total
orders.  So the device result equals this model bit for bit.  `recheck` rebuilds a witness from the definition with
the dense R of FeederTree.rmat()."""
import numpy as np

import network_ref as NR
import repair_ref as RR

TOPK = 32          # kCertTopK
MARGIN = 1e-12     # pu^2 in favour of "fits"


def _zone_arrays(hz, T):
    ev = np.asarray(hz["has_ev"]) > 0
    nmin = np.where(ev, RR.count_min(hz), 0)
    nmax = np.where(ev, RR.count_max(hz), 0)
    t = np.arange(T)[None, :]
    win = (t >= np.asarray(hz["start"])[:, None]) & (t < np.asarray(hz["end"])[:, None])
    if (ev & ((nmin > nmax) | (nmin > win.sum(axis=1)))).any():
        raise ValueError("a home's SOC target needs more hours than its plug-in window has")
    rating = np.asarray(hz["rating"], dtype=np.float64)
    if (ev & ~(np.isfinite(rating) & (rating >= 0.0))).any():
        raise ValueError("an EV home has a negative or non-finite rating")
    return ev & (nmin > 0), nmin, win, rating


def certify_zone(tr, hz, u, row_tol):
    """One zone: [kind, residence, step or k, need - cap] (int32), the kernels' rule."""
    load = np.asarray(hz["load"], dtype=np.float64)
    n, T = load.shape
    count, nmin, win, rating = _zone_arrays(hz, T)
    thr = row_tol + MARGIN
    if n == 0:
        return np.array([0, -1, -1, 0], dtype=np.int32)
    D0 = NR.zone_state(tr.parent, tr.r, tr.res_node, load)[1][np.asarray(tr.res_node, dtype=np.int64)]
    E = D0 - u
    j = int(np.argmax(E))                       # first maximum: lowest residence, then lowest step
    if E.flat[j] > thr:
        return np.array([1, j // T, j % T, 0], dtype=np.int32)
    hc = np.nonzero(count)[0]
    if hc.size == 0:
        return np.array([0, -1, -1, 0], dtype=np.int32)
    cols = RR._Columns(tr)
    A = np.stack([rating[h] * cols(int(h)) for h in hc], axis=1)        # [n residences, homes that count]
    K = min(TOPK, hc.size)
    top = np.argsort(-A, axis=1, kind="stable")[:, :K]                  # value descending, ties to the lowest home
    a = np.take_along_axis(A, top, axis=1)                              # [n, K]
    w = win[hc[top]]                                                    # [n, K, T]
    need = np.cumsum(nmin[hc[top]], axis=1)                             # [n, K]
    cap = np.zeros((n, K), dtype=np.int64)
    for k in range(1, K + 1):
        s = np.zeros((n, T))
        alive = np.ones((n, T), dtype=bool)
        m = np.zeros((n, T), dtype=np.int64)
        for r in range(k - 1, -1, -1):                                  # S_k in ascending order
            wr = w[:, r, :]
            s = s + np.where(wr, a[:, r, None], 0.0)                    # + 0.0 leaves s unchanged
            fits = (D0 + s) - u <= thr
            alive &= ~wr | fits
            m += alive & wr
        cap[:, k - 1] = m.sum(axis=1)
    d = need - cap
    j = int(np.argmax(d))                       # first maximum: lowest residence, then lowest k
    if d.flat[j] > 0:
        return np.array([2, j // K, j % K + 1, d.flat[j]], dtype=np.int32)
    return np.array([0, -1, -1, 0], dtype=np.int32)


def certify(zones, hm, vset=1.0, vhigh=1.05, row_tol=1e-9):
    """What Solver.certify_infeasible returns for the zones (FeederTree-like, solver order) and homes hm:
    dict(zone_cert [zones, 4] int32)."""
    u = vhigh * vhigh - vset * vset
    out, off = [], 0
    for tr in zones:
        s = slice(off, off + tr.n_res)
        out.append(certify_zone(tr, {k: np.asarray(v)[s] for k, v in hm.items()}, u, row_tol))
        off += tr.n_res
    return dict(zone_cert=np.array(out, dtype=np.int32).reshape(-1, 4))


def recheck(tr, hz, cert, vset=1.0, vhigh=1.05, row_tol=1e-9):
    """The witness of a certificate rebuilt from the definition with the dense R (FeederTree.rmat()): kind 1 returns
    the excess D0[i,t] - u - row_tol of the witness row; kind 2 returns need - cap of (i, k), each S_k member's
    charges counted greedily at every step of its window."""
    kind, i, x, _ = (int(v) for v in cert)
    u = vhigh * vhigh - vset * vset
    res = np.asarray(tr.res_node, dtype=np.int64)
    R = tr.rmat()[np.ix_(res, res)]
    load = np.asarray(hz["load"], dtype=np.float64)
    D0 = R[i] @ load
    if kind == 1:
        return D0[x] - u - row_tol
    assert kind == 2
    count, nmin, win, rating = _zone_arrays(hz, load.shape[1])
    hc = np.nonzero(count)[0]
    a = rating[hc] * R[i, hc]
    S = hc[sorted(range(hc.size), key=lambda j: (-a[j], hc[j]))[:x]]
    cap = 0
    for t in range(load.shape[1]):
        c = np.sort(rating[S[win[S, t]]] * R[i, S[win[S, t]]])
        cap += int(np.searchsorted(D0[t] + np.cumsum(c) - u, row_tol + MARGIN, side="right"))
    return int(nmin[S].sum()) - cap

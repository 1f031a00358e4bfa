"""Host model (numpy, plain loops) of the large-zone operator kernel csrc/tree_newton.cu.

Test infrastructure: it restates the DEVICE algorithm so that its linear algebra can be checked against
dense matrices without a GPU; the product never imports it.

Reference problem: class Utility (lpsolver.py:163-238), one hour of it:
    min 1/2 |g - z|^2   s.t.  g >= 0,  R g <= u,        R = 2 F D F^T   (compute_Rmat, lpsolver.py:17-26).
For a radial zone R is never needed as a matrix.  With rho_k = 2 r_k on the edge above node k,
    (R x)_k = mu_k,   mu_k = mu_parent + rho_k Lam_k,   Lam_k = x_k + sum_{children c} Lam_c
(one pass leaves -> root for the subtree sums, one pass root -> leaves for the potentials), and the linear
system of one active-set guess -- rows A at their limit on the piece F = {g > 0},
    R_AF (z_F - R_FA x_A) - s x_A = t_A
-- is a two-point boundary problem on the same tree: every subtree answers its parent's (mu, v) with the
affine map (Lam, f) = M (mu, v) + m, maps add over the children, a node is eliminated with one 2x2 solve.
"""
import numpy as np


def tree_product(parent, rho, x):
    """R_full x over ALL nodes of the tree (x on nodes, 0 where no injection)."""
    n = len(parent)
    lam = np.array(x, dtype=float)
    for k in range(n - 1, -1, -1):
        if parent[k] >= 0:
            lam[parent[k]] += lam[k]
    mu = np.zeros(n)
    for k in range(n):
        mu[k] = (mu[parent[k]] if parent[k] >= 0 else 0.0) + rho[k] * lam[k]
    return mu


def tree_solve(parent, rho, z, F, A, t, s):
    """x on the nodes of A (0 elsewhere) with  v_k - s x_k = t_k  for k in A, where
    g = (z - R x) on F, 0 elsewhere, v = R g.  Returns (x, mu = R x, g, v).  O(nodes)."""
    n = len(parent)
    S = np.zeros((n, 2, 2))
    sv = np.zeros((n, 2))
    keep = [None] * n
    for k in range(n - 1, -1, -1):
        r = rho[k]
        phi = 1.0 if F[k] else 0.0
        Sp = S[k].copy()
        Sp[1, 0] -= phi
        sp = sv[k].copy()
        sp[1] += phi * z[k]
        if not A[k]:
            # a = (mu_k, v_k) = B (p + r sp),  (Lam, f) = Sp a + sp
            B = np.linalg.inv(np.eye(2) - r * Sp)
            M = Sp @ B
            m = B @ sp
            keep[k] = (B, r * (B @ sp))
        else:
            Q = np.array([[1.0 - r * Sp[0, 0], -r * (1.0 + Sp[0, 1] * s)],
                          [-r * Sp[1, 0], s * (1.0 - r * Sp[1, 1])]])
            q0 = np.array([r * sp[0] + r * Sp[0, 1] * t[k], -t[k] + r * Sp[1, 1] * t[k] + r * sp[1]])
            Qi = np.linalg.inv(Q)
            C = np.array([[Sp[0, 0], 1.0 + Sp[0, 1] * s], [Sp[1, 0], Sp[1, 1] * s]])
            c0 = np.array([Sp[0, 1] * t[k] + sp[0], Sp[1, 1] * t[k] + sp[1]])
            M = C @ Qi
            m = C @ (Qi @ q0) + c0
            keep[k] = (Qi, Qi @ q0)
        if parent[k] >= 0:
            S[parent[k]] += M
            sv[parent[k]] += m
    mu = np.zeros(n)
    v = np.zeros(n)
    x = np.zeros(n)
    for k in range(n):
        p = np.array([mu[parent[k]], v[parent[k]]]) if parent[k] >= 0 else np.zeros(2)
        Mk, mk = keep[k]
        a = Mk @ p + mk
        if A[k]:
            mu[k], x[k] = a
            v[k] = t[k] + s * x[k]
        else:
            mu[k], v[k] = a
    g = np.where(F, z - mu, 0.0)
    return x, mu, g, v


# ------------------------------------------------------------------------------------------------------------------
# The same operations level by level (what a CTA does: one thread per node of a level, one barrier per level), and the
# projection built on them.  Nodes are renumbered breadth-first: a level is a contiguous range, the children of a node
# are contiguous in the next level.  Two things make the elimination robust on real feeders:
#
#   * edges of (numerically) zero resistance are contracted before anything else -- the reference's network 121144 has
#     primary edges of 1e-20 -- so a node can carry several residences; their voltage rows are identical, the node has
#     ONE row and one multiplier, its homes differ only in z and in whether they are on the piece;
#   * an active row whose subtree holds no home of the piece has no leverage of its own (nothing below it flows, its
#     voltage is its parent's): its 2 x 2 pivot would be the shift alone.  Such a node PINS its parent instead --
#     "your voltage is my target" -- and hands its multiplier up as the parent's unknown; pins travel up idle chains,
#     the first of several pins on a node is kept and the others (duplicate rows) sit the guess out.

HESS_SHIFT = 1e-20        # relative diagonal shift: structural singularities are handled by the pins, not by the shift
ARC_MIN = 2.0 ** -20
PDAS_MAX = 24
PHI_NOISE = 1e-14
CONTRACT_REL = 1e-10      # edges below this fraction of the largest root-to-node resistance are contracted
DEG_TOL = 1e-9           # |d(flow of the subtree)/d(mu)| below this: no home of the piece below an effective row
PDAS_SLACK = 1e-13        # a row off the guess re-enters when it is violated by more than this fraction of u
SKYLINE_OUTER = 32        # from this outer iteration on, every violated row is a working row (not only the skyline)


def contract_tree(parent, r, res_node, rel=CONTRACT_REL):
    """Merge every node whose edge resistance is negligible into its parent.  Returns (parent', r', res_node', keep)."""
    parent = np.asarray(parent)
    r = np.asarray(r, dtype=float)
    n = len(parent)
    cum = np.zeros(n)
    for k in range(n):
        cum[k] = (cum[parent[k]] if parent[k] >= 0 else 0.0) + r[k]
    tiny = (r <= rel * cum.max()) & (parent >= 0)
    rep = np.arange(n)
    for k in range(n):
        if tiny[k]:
            rep[k] = rep[parent[k]]
    keep = np.nonzero(~tiny)[0]
    new = np.full(n, -1)
    new[keep] = np.arange(len(keep))
    par2 = np.where(parent[keep] >= 0, new[rep[np.maximum(parent[keep], 0)]], -1)
    return par2, r[keep], new[rep[np.asarray(res_node)]], keep


class LevelTree:
    def __init__(self, parent, r, res_node, contract=True):
        if contract:
            parent, r, res_node, _ = contract_tree(parent, r, res_node)
        parent = np.asarray(parent)
        n = len(parent)
        depth = np.zeros(n, dtype=np.int64)
        for k in range(n):
            depth[k] = depth[parent[k]] + 1 if parent[k] >= 0 else 0
        order_lv = []
        new = np.full(n, -1, dtype=np.int64)
        cnt = 0
        for d in range(depth.max() + 1):
            nodes = np.nonzero(depth == d)[0]
            if d > 0:
                nodes = nodes[np.argsort(new[parent[nodes]], kind="stable")]
            new[nodes] = cnt + np.arange(len(nodes))
            cnt += len(nodes)
            order_lv.append(nodes)
        order = np.concatenate(order_lv)
        self.order = order                      # new index -> node of the contracted tree
        self.n = n
        self.parent = np.where(parent[order] >= 0, new[np.maximum(parent[order], 0)], -1)
        self.rho = 2.0 * np.asarray(r, dtype=float)[order]
        dep = depth[order]
        self.lvl = np.searchsorted(dep, np.arange(dep.max() + 2))          # level offsets
        self.child0 = np.zeros(n, dtype=np.int64)
        self.nchild = np.zeros(n, dtype=np.int64)
        for k in range(n - 1, -1, -1):
            p = self.parent[k]
            if p >= 0:
                self.child0[p] = k
                self.nchild[p] += 1
        self.res = new[np.asarray(res_node)]    # node (new index) of every home
        self.nhome = np.bincount(self.res, minlength=n)
        self.isres = self.nhome > 0

    def levels_up(self):
        return [(self.lvl[l], self.lvl[l + 1]) for l in range(len(self.lvl) - 2, -1, -1)]

    def levels_down(self):
        return [(self.lvl[l], self.lvl[l + 1]) for l in range(len(self.lvl) - 1)]

    def _child_sum(self, a, lo, hi):
        out = np.zeros((hi - lo,) + a.shape[1:])
        c0, nc = self.child0[lo:hi], self.nchild[lo:hi]
        for j in range(int(nc.max()) if hi > lo else 0):
            m = nc > j
            out[m] += a[c0[m] + j]
        return out

    def product(self, x):
        """R x on all nodes (x on nodes)."""
        lam = np.array(x, dtype=float)
        for lo, hi in self.levels_up():
            lam[lo:hi] += self._child_sum(lam, lo, hi)
        mu = np.zeros(self.n)
        for lo, hi in self.levels_down():
            p = self.parent[lo:hi]
            mu[lo:hi] = np.where(p >= 0, mu[np.maximum(p, 0)], 0.0) + self.rho[lo:hi] * lam[lo:hi]
        return mu

    def solve(self, nF, zF, A, t, s):
        """One active-set guess.  nF[k] / zF[k]: number of homes of node k on the piece / sum of their targets;
        A: active node rows; t: their targets; s: shift.  x on A (0 elsewhere) with v - s x = t on the rows that take
        part, for g_h = z_h - mu[node(h)] on the piece, v = R g.  Returns (x, mu, v)."""
        n = self.n
        M = np.zeros((n, 4))                    # map of the subtree with the node NOT enforcing a row: (Lam, f) = M (mu_p, v_p) + m
        m = np.zeros((n, 2))
        K = np.zeros((n, 4))                    # back-substitution of the node as it finally acts
        kv = np.zeros((n, 2))
        Kn = np.zeros((n, 4))                   # ... and as a plain node (a pinning node whose pin is not kept)
        kvn = np.zeros((n, 2))
        pin = np.zeros(n, dtype=bool)           # node pins its parent
        tauP = np.full(n, np.inf)               # ... to this voltage
        P4 = np.zeros((n, 4))                   # pinning node: S00, S01, s0 of its dual flow, constant primal flow c
        tau = np.full(n, np.inf)                # target of the effective row of the node
        src = np.full(n, -2, dtype=np.int64)    # -2: no effective row, -1: own row, >= 0: the child whose pin is kept

        def plain(S, sv, r):
            a_, b_, c_, d_ = 1.0 - r * S[0], -r * S[1], -r * S[2], 1.0 - r * S[3]
            inv = 1.0 / (a_ * d_ - b_ * c_)
            i = (d_ * inv, -b_ * inv, -c_ * inv, a_ * inv)
            q0, q1 = r * sv[0], r * sv[1]
            k0, k1 = i[0] * q0 + i[1] * q1, i[2] * q0 + i[3] * q1
            Mk = (S[0] * i[0] + S[1] * i[2], S[0] * i[1] + S[1] * i[3], S[2] * i[0] + S[3] * i[2], S[2] * i[1] + S[3] * i[3])
            mk = (S[0] * k0 + S[1] * k1 + sv[0], S[2] * k0 + S[3] * k1 + sv[1])
            return Mk, mk, i, (k0, k1)

        def active(S, sv, r, tk):
            a_, c_ = 1.0 - r * S[0], -r * S[2]
            b_, d_ = -r * (1.0 + S[1] * s), s * (1.0 - r * S[3])
            q0, q1 = r * (sv[0] + S[1] * tk), -tk + r * (S[3] * tk + sv[1])
            C01, C11, c00, c01 = 1.0 + S[1] * s, S[3] * s, S[1] * tk + sv[0], S[3] * tk + sv[1]
            inv = 1.0 / (a_ * d_ - b_ * c_)
            i = (d_ * inv, -b_ * inv, -c_ * inv, a_ * inv)
            k0, k1 = i[0] * q0 + i[1] * q1, i[2] * q0 + i[3] * q1
            Mk = (S[0] * i[0] + C01 * i[2], S[0] * i[1] + C01 * i[3], S[2] * i[0] + C11 * i[2], S[2] * i[1] + C11 * i[3])
            mk = (S[0] * k0 + C01 * k1 + c00, S[2] * k0 + C11 * k1 + c01)
            return Mk, mk, i, (k0, k1)

        for lo, hi in self.levels_up():
            for k in range(lo, hi):             # (scalar here; one thread per node on the device)
                tk, sk = (t[k], -1) if A[k] else (np.inf, -2)
                kids = range(self.child0[k], self.child0[k] + self.nchild[k])
                for c in kids:
                    if pin[c] and tauP[c] < tk:
                        tk, sk = tauP[c], c
                Sn = np.zeros(4); mn = np.zeros(2); Se = np.zeros(4); me = np.zeros(2)
                for c in kids:
                    Sn += M[c]; mn += m[c]
                    if c == sk:
                        me[1] += P4[c, 3]
                    else:
                        Se += M[c]; me += m[c]
                for S, sv in ((Sn, mn), (Se, me)):
                    S[2] -= nF[k]
                    sv[1] += zF[k]
                r = self.rho[k]
                M[k], m[k], Kn[k], kvn[k] = plain(Sn, mn, r)
                K[k], kv[k] = Kn[k], kvn[k]
                tau[k], src[k] = tk, sk
                if sk == -2:
                    continue
                if abs(Se[2]) < DEG_TOL:
                    # nothing below responds to the multiplier: the row pins the parent (no parent: it cannot bind)
                    if self.parent[k] < 0:
                        src[k] = -2
                        continue
                    c = Se[3] * tk + me[1]
                    pin[k] = True
                    tauP[k] = tk - r * c
                    P4[k] = (Se[0], Se[1], me[0], c)
                else:
                    M[k], m[k], K[k], kv[k] = active(Se, me, r, tk)
        mu = np.zeros(n)
        v = np.zeros(n)
        x = np.zeros(n)
        xi_in = np.full(n, np.nan)              # dual flow handed down to the node whose pin was kept (nan: not kept)
        for lo, hi in self.levels_down():
            for k in range(lo, hi):
                p = self.parent[k]
                mp, vp = (mu[p], v[p]) if p >= 0 else (0.0, 0.0)
                if pin[k]:
                    if np.isnan(xi_in[k]):      # the parent kept another pin (or was dropped itself): a plain node
                        mu[k] = Kn[k, 0] * mp + Kn[k, 1] * vp + kvn[k, 0]
                        v[k] = Kn[k, 2] * mp + Kn[k, 3] * vp + kvn[k, 1]
                        continue
                    mu[k] = mp + self.rho[k] * xi_in[k]
                    v[k] = tau[k]
                    xi = xi_in[k] - (P4[k, 0] * mu[k] + P4[k, 1] * v[k] + P4[k, 2])
                elif src[k] != -2:
                    mu[k] = K[k, 0] * mp + K[k, 1] * vp + kv[k, 0]
                    xi = K[k, 2] * mp + K[k, 3] * vp + kv[k, 1]
                    v[k] = tau[k] + s * xi
                else:
                    mu[k] = K[k, 0] * mp + K[k, 1] * vp + kv[k, 0]
                    v[k] = K[k, 2] * mp + K[k, 3] * vp + kv[k, 1]
                    continue
                if src[k] == -1:
                    x[k] = xi
                else:
                    xi_in[src[k]] = xi
        return x, mu, v

    def project(self, z_res, u, lam0_res=None, tol=1e-11, maxit=200, stats=None):
        """argmin 1/2 |g - z|^2, g >= 0, R g <= u over the residences of the zone (z_res in home order).
        Same iteration as oracle.project_voltage (piece minimised exactly by a primal-dual active set, line search of
        the dual, Levenberg-Marquardt safeguard) with every linear-algebra step done on the tree.  Returns (g, lam, its);
        lam sits on the first home of every node."""
        n, res = self.n, self.res
        isres = self.isres
        z = np.asarray(z_res, dtype=float)
        lam = np.zeros(n)
        if lam0_res is not None:
            np.add.at(lam, res, np.maximum(lam0_res, 0.0))
        ones = self.product(self.nhome.astype(float))
        scale = float((self.nhome * ones * ones).sum()) / max(len(res), 1) ** 2
        nsolve = nprod = 0

        def node_sum(x_h):
            return np.bincount(res, weights=x_h, minlength=n)

        def phi(lm):
            gg = np.maximum(z - self.product(lm)[res], 0.0)
            return 0.5 * gg @ gg + u * lm.sum(), gg

        f, g = phi(lam)
        nprod += 1
        tau = 1.0
        for it in range(maxit):
            v = self.product(node_sum(g))
            nprod += 1
            grad = np.where(isres, u - v, np.inf)
            kkt = np.max(np.abs(np.where(lam > 0, grad, np.minimum(grad, 0.0))))
            if kkt < tol:
                if stats is not None:
                    stats.update(solves=nsolve, products=nprod, outer=it, active=int((lam > 0).sum()))
                lam_h = np.zeros(len(res))
                first = np.unique(res, return_index=True)[1]
                lam_h[first] = lam[res[first]]
                return g, lam_h, it
            # working rows: the multipliers' support and the SKYLINE of the violated rows -- a violated row enters when no row
            # in the subtree of its parent is more violated.  Under a heavy shared drop thousands of rows are violated by
            # similar amounts, a hundred end up binding; holding the skyline repairs most of the others, the rest is admitted
            # by the next iteration (the KKT test always runs over all rows).  Siblings share their parent's subtree, so the
            # skyline admits one row per node per iteration; after SKYLINE_OUTER iterations every violated row enters.
            viol = np.where(isres, np.maximum(-grad, 0.0), 0.0)
            sub = viol.copy()
            for lo, hi in self.levels_up():
                c0, nc = self.child0[lo:hi], self.nchild[lo:hi]
                for j in range(int(nc.max()) if hi > lo else 0):
                    m = nc > j
                    sub[lo:hi][m] = np.maximum(sub[lo:hi][m], sub[c0[m] + j])
            ref = np.where(self.parent >= 0, sub[np.maximum(self.parent, 0)], sub)
            W = isres & ((lam > 0) | ((viol > 0) & ((viol >= ref) | (it >= SKYLINE_OUTER))))
            Fh = g > 0
            nF = node_sum(Fh.astype(float))
            zF = node_sum(np.where(Fh, z, 0.0))
            shift = HESS_SHIFT * scale + 1e-300
            t = u - shift * lam
            A = W.copy()
            ok = False
            for _ in range(PDAS_MAX):
                x, mu_x, vx = self.solve(nF, zF, A, t, shift)
                nsolve += 1
                bad_in = A & (x <= 0)
                bad_out = W & ~A & (u - vx - shift * lam < -PDAS_SLACK * u)
                if not bad_in.any() and not bad_out.any():
                    ok = True
                    break
                A = (A & ~bad_in) | bad_out
            # line search on the segment to the minimiser; guesses that did not settle: the last one, clipped, is tried first
            settled = ok
            d = np.where(W, np.maximum(x, 0.0) - lam, 0.0)
            slope = float(np.where(W, grad, 0.0) @ d)
            a = 1.0
            ok = False
            while slope < 0.0 and a >= (ARC_MIN if settled else 1.0 / 64.0):
                ln = np.maximum(lam + a * d, 0.0)
                fn, gn = phi(ln)
                nprod += 1
                if fn <= f + 1e-4 * a * slope + PHI_NOISE * abs(f):
                    ok = True
                    break
                a *= 0.5
            if not ok:
                eps = min(1e-8, kkt)
                free = W & ~((lam <= eps) & (grad > 0))
                rest = W & ~free
                zt = z - self.product(np.where(rest, lam, 0.0))[res] if (lam[rest] > 0).any() else z
                zFt = node_sum(np.where(Fh, zt, 0.0))
                while True:
                    sg = max(HESS_SHIFT, 1e-12) * tau * scale + 1e-300
                    x, _, _ = self.solve(nF, zFt, free, u - sg * lam, sg)
                    nsolve += 1
                    d = np.where(free, x - lam, np.where(W, -lam, 0.0))
                    a, found = 1.0, False
                    while a >= ARC_MIN:
                        ln = np.maximum(lam + a * d, 0.0)
                        fn, gn = phi(ln)
                        nprod += 1
                        if fn <= f + 1e-4 * float(np.where(W, grad, 0.0) @ (ln - lam)) + PHI_NOISE * abs(f):
                            found = True
                            break
                        a *= 0.5
                    if found or tau > 1e40:
                        break
                    tau *= 1e3
                if a == 1.0:
                    tau = max(1.0, tau / 10.0)
            lam, f, g = ln, fn, gn
        raise RuntimeError("tree projection did not converge (kkt=%g)" % kkt)

"""numpy model of one iteration of the device ADMM loop (tests/test_gpu_admm_steps.py).

One iteration k -> k+1 takes (P_est[k], P_sch[k], Gamma[k]) and is three exact operations:
    home solve      P_sch[k+1], P_ev[k+1] = the homes' selections (revs_oracle.home_subproblem, home_solve.cu)
    operator QP     P_est[k+1] = argmin 1/2 |g - z|^2  s.t.  g >= 0, R g <= u  in every (zone, step) column,
                    z = next_target(P_est[k], P_sch[k], Gamma[k])
    dual update     Gamma[k+1] = Gamma[k] + kappa/2 (P_est[k+1] - P_sch[k+1]), diff[k+1] = |P_est[k+1] - P_sch[k+1]| / T
`next_target`, `dual_update` and `homes` round every operation as the kernels do (dual_update.cu, home_solve.cu), so
they equal the device's values bit for bit on equal inputs.  The projection is not restated: `certify_projection`
proves that a given g is the projection, whatever computed it, with nothing but the KKT conditions."""
import numpy as np
from scipy.optimize import linprog

import revs_oracle as O


def next_target(P_est, P_sch, Gamma, kappa):
    """z of the next operator QP, in the order of dual_update.cu: (e + s) * 0.5 - Gamma / kappa."""
    return (P_est + P_sch) * 0.5 - Gamma / kappa


def dual_update(Gamma, P_est1, P_sch1, kappa):
    """(Gamma[k+1], diff[k+1]): Gamma + (0.5 kappa) (P_est1 - P_sch1), and sqrt(sum_t check^2) / T per home.  The sum of
    squares is taken in extended precision, so the device's sum (lane-wise fma, then a shuffle tree) is the only
    rounding left in a comparison."""
    check = P_est1 - P_sch1
    G = Gamma + (0.5 * kappa) * check
    sq = (check.astype(np.longdouble) ** 2).sum(axis=1)
    return G, np.sqrt(sq.astype(np.float64)) / check.shape[1]


def homes(cost, hm, P_est, P_sch, Gamma, kappa):
    """(P_sch [H,T], P_ev [H,T], SOC [H,T+1]) of the home solve from the previous iterates, home by home."""
    load = np.asarray(hm["load"], dtype=np.float64)
    H, T = load.shape
    P_sch1, P_ev, SOC = np.empty((H, T)), np.zeros((H, T)), np.zeros((H, T + 1))
    for i in range(H):
        ev = {}
        if hm["has_ev"][i]:
            ev = dict(rating=hm["rating"][i], capacity=hm["capacity"][i], initial=hm["initial"][i],
                      start=hm["start"][i], end=hm["end"][i])
        P_ev[i], SOC[i], P_sch1[i] = O.home_subproblem(cost, load[i], ev, P_est[i], P_sch[i], Gamma[i], kappa)
    return P_sch1, P_ev, SOC


def _multipliers_lstsq(RF, r):
    """lam >= 0 with R_FA lam = r by least squares on every candidate row (the minimum-norm solution shares lam
    between identical rows); None when it is not non-negative."""
    if RF.shape[0] == 0:
        return np.zeros(RF.shape[1])
    lam = np.linalg.lstsq(RF, r, rcond=None)[0]
    return lam if lam.min() >= 0.0 else None


def _multipliers_lp(RF, r, RZ, zZ, tol):
    """min s  s.t. |r - R_FA lam| <= s, z_Z - R_ZA lam <= tol / 2, lam >= 0.  The columns of R_FA are scaled to a largest
    entry of 1 so that HiGHS sees coefficients of order one; its tolerances only steer the search, the caller
    checks the multipliers it returns exactly."""
    m = RF.shape[1]
    c = np.maximum(np.vstack([RF, RZ]).max(axis=0), 1e-300)
    MF, MZ = RF / c, RZ / c
    nF, nZ = MF.shape[0], MZ.shape[0]
    A = np.zeros((2 * nF + nZ, m + 1))
    A[:nF, :m], A[:nF, m] = MF, -1.0
    A[nF:2 * nF, :m], A[nF:2 * nF, m] = -MF, -1.0
    A[2 * nF:, :m] = -MZ
    b = np.concatenate([r, -r, 0.5 * tol - zZ])        # half of tol: a vertex ON the bound lands past it after rounding
    obj = np.zeros(m + 1)
    obj[m] = 1.0
    res = linprog(obj, A_ub=A, b_ub=b, bounds=[(0.0, None)] * (m + 1), method="highs",
                  options=dict(primal_feasibility_tolerance=1e-10, dual_feasibility_tolerance=1e-10))
    if res.x is None:
        return None
    return np.maximum(res.x[:m], 0.0) / c


def _residual(RA, z, g, lam, F):
    """Largest violation of the KKT conditions by lam >= 0 on the candidate rows: |g_F - (z_F - R_FA lam)| on the
    homes with g > 0, z_j - R_jA lam on the homes at zero."""
    w = z - RA @ lam
    out = np.abs(g[F] - w[F]).max() if F.any() else 0.0
    if (~F).any():
        out = max(out, w[~F].max())
    return out


def certify_projection(R, z, g, u, tol=1e-9, use_lstsq=True):
    """Prove, column by column, that g [n,T] is the Euclidean projection of z [n,T] onto {g >= 0, R g <= u}.

    A column is certified when g >= 0, R g <= u + tol, and some lam >= 0 on the candidate rows
    A = {i : (R g)_i >= u - tol} gives g_j = z_j - (R_jA lam) within tol where g_j > 0 and z_j - R_jA lam <= tol where
    g_j = 0.  These are the KKT conditions of a strictly convex QP, so a certified g is its unique solution (up to
    tol), whatever computed it; the device's own multipliers are not used.  lam comes from least squares on all
    candidate rows when that is non-negative, else from a small LP (identical rows of R -- residences on one node --
    make lam non-unique, where least squares or NNLS may pick one that breaks the g = 0 side).  Columns without a
    candidate row must satisfy g == max(z, 0) to 1e-12.

    Returns dict(ok [T] bool, resid [T] (the certificate's residual: the largest infeasibility, KKT violation or
    |g - [z]_+|), rows [T] (candidate rows), lp (columns that needed the LP))."""
    R = np.asarray(R, dtype=np.float64)
    z = np.asarray(z, dtype=np.float64).reshape(R.shape[0], -1)
    g = np.asarray(g, dtype=np.float64).reshape(R.shape[0], -1)
    T = z.shape[1]
    V = R @ g
    over = np.maximum((V - u).max(axis=0, initial=-np.inf), 0.0)
    neg = (g < 0.0).any(axis=0)
    cand = V >= u - tol
    rows = cand.sum(axis=0)
    resid = np.where(rows == 0, np.abs(g - np.maximum(z, 0.0)).max(axis=0, initial=0.0), 0.0)
    ok = (rows == 0) & (resid <= 1e-12)
    lp = 0
    for t in np.nonzero(rows > 0)[0]:
        A = cand[:, t]
        RA = R[:, A]
        F = g[:, t] > 0.0
        r = z[F, t] - g[F, t]
        best = np.inf
        lam = _multipliers_lstsq(RA[F], r) if use_lstsq else None
        if lam is not None:
            best = _residual(RA, z[:, t], g[:, t], lam, F)
        if best > tol:
            lp += 1
            lam = _multipliers_lp(RA[F], r, RA[~F], z[~F, t], tol)
            if lam is not None:
                best = min(best, _residual(RA, z[:, t], g[:, t], lam, F))
        resid[t] = best
        ok[t] = best <= tol
    resid = np.maximum(resid, np.maximum(over, np.maximum(-g.min(axis=0, initial=0.0), 0.0)))
    ok &= (over <= tol) & ~neg
    return dict(ok=ok, resid=resid, rows=rows, lp=lp)

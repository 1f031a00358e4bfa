"""Every iteration of the device ADMM loop checked on its own, from the state the device itself left behind.

The trajectory tests compare whole runs with the oracle, which runs the same algorithm, within tolerances loose
enough for errors that add up along a trajectory.  Here iteration k+1 is recomputed from (P_est[k], P_sch[k],
Gamma[k]) as read back from the device (tests/admm_step_ref.py):
    home solve    P_sch[k+1], P_ev[k+1] and SOC bit for bit (home_solve_kernel<SLOTS>, iterative pick and ranking)
    operator QP   P_est[k+1] is the projection of z = next_target(...) in every (zone, step) column, proved by a KKT
                  certificate that does not use the device's multipliers (warp kernels, CTA classes, tree-Newton,
                  in-loop screening, warm-started working sets)
    dual update   Gamma[k+1] bit for bit, diff[k+1] to 1e-14 relative (dual_update_kernel<SLOTS, DSUM>)
    download      the charging bit masks are P_ev > 0 packed LSB first in 64-step words, zero past T, and
                  expand_schedule rebuilds results()'s P_ev and SOC from them exactly
and the captured graph (solve_admm) reproduces the stepped state after every k.  A failure names the case, the
iteration, the zone and the column or home.  The cases sit on the size and horizon boundaries where the kernels
switch: zone-size classes at T = 24, horizons 1..256 (SLOTS of the home solve and the dual update, shared-memory
opt-in, mask words, both in-loop screening kernels), windows and charge counts that run both selection paths."""
import numpy as np
import pytest

import admm_step_ref as AR
import revs_oracle as O
from revs_admm_b200 import expand_schedule
from test_gpu_edges import _problem
from test_gpu_newton_shapes import deep, odd_wide, wide2

pytestmark = pytest.mark.gpu

TOL = 1e-9           # certificate tolerance, kW and pu^2


def _vary_homes(hm, T, seed):
    """Per-home plug-in windows and charge counts.  Windows cycle through [0, T), ones that end at T, ones of exactly
    n_min steps, ones that cross the 32-step lane boundary and the population's own; every other group of five
    homes needs more than 24 charging steps at most (full ranking in home_solve_kernel), the rest at most 24
    (iterative pick).  (n_min, n_max) are set through capacity and initial SOC; n_min = 0 (initial SOC >= 0.9)
    comes up with the draw.  Every seventh home has a flat load, so that equal tariff steps tie exactly."""
    rng = np.random.default_rng(seed)
    H = len(hm["load"])
    out = {k: np.array(v, copy=True) for k, v in hm.items()}
    for i in range(H):
        ranking = (i // 5) % 2 == 1
        M = int(rng.integers(25, 41)) if ranking else int(rng.integers(1, 25))
        kind = i % 5
        st, en = int(hm["start"][i]), int(hm["end"][i])
        if kind == 0 or not (0 <= st < en <= T):
            st, en = 0, T
        if kind == 1:
            st = T - int(rng.integers(1, T + 1))
            en = T
        elif kind == 2:
            L = int(rng.integers(1, min(T, M) + 1))
            st = int(rng.integers(0, T - L + 1))
            en = st + L
        elif kind == 3 and T > 32:
            st, en = int(rng.integers(12, 32)), int(rng.integers(33, min(T, 60) + 1))
        L = en - st
        m = L if kind == 2 else int(rng.integers(0, min(L, M) + 1))
        M = max(M, m)
        while m > 0 and m - 0.5 > 9.0 * (M - m + 1):      # keep the initial SOC >= 0
            M += 1
        if m == 0:
            step, init = 0.05 / (M + 0.5), 0.95
        else:
            step = 0.1 / (M - m + 1)
            init = 0.9 - (m - 0.5) * step
        out["start"][i], out["end"][i] = st, en
        out["capacity"][i] = out["rating"][i] / step
        out["initial"][i] = init
        if i % 7 == 3:
            out["load"][i] = 0.5
    return out


def _counts(hm):
    return [O.count_window(hm["rating"][i], hm["capacity"][i], hm["initial"][i]) for i in range(len(hm["load"]))]


def _case(name):
    """(sizes, T, trees, homes, tariff, kw, iterations, options)."""
    from revs_admm_b200.feeder import synthetic_homes, synthetic_tariff
    kw = dict(kappa=5.0, vset=1.0, vlow=0.95, vhigh=1.02)
    classes = {"cls_warp_small": [1, 16, 17, 127, 128, 129, 192], "cls_warp_big": [193, 255, 256, 257, 320],
               "cls_cta": [321, 512, 513, 700]}
    if name in classes:
        sizes, T = classes[name], 24
        trees, hm, cost = _problem(sizes, T, seed=sum(sizes))
        if name == "cls_cta":       # up to ~80 binding rows: beyond the first CTA class, within the dense kernels' 128
            return sizes, T, trees, hm, cost, dict(kw, vhigh=1.04), 4, dict(newton_min_n=4096)
        return sizes, T, trees, hm, cost, kw, 5, dict(newton_min_n=4096)
    if name == "newton":
        sizes, T = [600, 90], 24
        trees, hm, cost = _problem(sizes, T, seed=690)
        return sizes, T, trees, hm, cost, dict(kw, vhigh=1.05), 5, {}
    if name in ("newton_wide", "newton_deep", "newton_odd"):    # layout branches of the tree-Newton kernel
        tr, K = {"newton_wide": (wide2(), 5), "newton_deep": (deep(1025), 3), "newton_odd": (odd_wide(), 5)}[name]
        T = 24
        hm = synthetic_homes(tr.n_res, T, seed=tr.n_res)
        return [tr.n_res], T, [tr], hm, synthetic_tariff(T), kw, K, dict(newton_min_n=0)
    if name == "handover":          # every charger free in every step: working sets beyond 16 and 32 rows
        sizes, T = [120, 96], 12
        trees, hm, cost = _problem(sizes, T, seed=77, r_secondary=2e-3, adoption=1.0)
        hm["start"][:] = 0
        hm["end"][:] = T
        return sizes, T, trees, hm, cost, kw, 4, dict(newton_min_n=4096)
    if name == "no_warp":
        sizes, T = [40, 150, 300], 24
        trees, hm, cost = _problem(sizes, T, seed=490)
        return sizes, T, trees, hm, cost, kw, 5, dict(warp_kernel=0, newton_min_n=4096)
    if name == "padding":           # 133 homes, zones of 37, 91 and 5: padding rows in every 32-home tile and in Hp
        sizes, T = [37, 91, 5], 40
        trees, hm, cost = _problem(sizes, T, seed=133)
        return sizes, T, trees, _vary_homes(hm, T, 133), cost, kw, 5, {}
    # horizons: "T<n>" or "T<n>_noscreen"
    T = int(name[1:].split("_")[0])
    sizes = [40, 150]
    trees, hm, cost = _problem(sizes, T, seed=1000 + T)
    opts = dict(screen=0) if name.endswith("noscreen") else {}
    return sizes, T, trees, _vary_homes(hm, T, T), cost, kw, 3 if T >= 192 else 5, opts


HORIZONS = [1, 31, 32, 33, 64, 65, 96, 97, 128, 129, 185, 191, 192, 256]      # 185..191: dual_update opts in to > 48 KB of shared memory
CASES = ["cls_warp_small", "cls_warp_big", "cls_cta", "newton", "newton_wide", "newton_deep", "newton_odd", "handover", "no_warp", "padding"] + \
        [f"T{T}" for T in HORIZONS] + ["T96_noscreen", "T97_noscreen"]


def _pack(P_ev):
    """P_ev > 0 as bit masks [H, ceil(T/64)]: step t is bit t % 64 of word t // 64, bits past T are zero."""
    H, T = P_ev.shape
    W = (T + 63) // 64
    bits = np.zeros((H, 64 * W), dtype=np.uint64)
    bits[:, :T] = P_ev > 0.0
    return (bits.reshape(H, W, 64) << np.arange(64, dtype=np.uint64)).sum(axis=2, dtype=np.uint64)


def _run(lib, sizes, T, trees, hm, cost, kw, K, opts):
    """K stepped iterations with every output read back after each, then solve_admm(iter_max=k) on the same solver."""
    steps, graph = [], []
    with lib.Solver(sizes, T) as s:
        for k, v in opts.items():
            s.set_option(k, v)
        s.set_feeder_trees(trees)
        s.set_homes(**hm)
        s.set_tariff(cost)
        s.admm_begin(iter_max=K, **kw)
        for k in range(K):
            s.admm_step()
            st = s.results(k + 1)
            st["P_est"], st["Gamma"] = s.estimate()
            st["compact"] = s.schedule_compact()
            steps.append(st)
        stats = s.stats()
        for k in range(1, K + 1):
            assert s.solve_admm(iter_max=k, **kw) == k
            g = s.results(k)
            g["P_est"], g["Gamma"] = s.estimate()
            graph.append(g)
    return steps, graph, stats


def _first(mask):
    idx = np.argwhere(mask)
    return [tuple(int(v) for v in i) for i in idx[:4]], int(mask.sum())


def check_steps(name, sizes, Rz, hm, cost, kw, steps):
    """Every iteration of `steps` (dicts of P_sch, P_ev, SOC, diff, P_est, Gamma, compact) against the model, each
    from the previous one's state.  Returns (certified columns with candidate rows, columns that needed the LP)."""
    H, T = hm["load"].shape
    kappa = kw["kappa"]
    u = kw["vhigh"] ** 2 - kw["vset"] ** 2
    off = np.concatenate([[0], np.cumsum(sizes)])
    ev = hm["has_ev"].astype(bool)
    prev = (np.zeros((H, T)),) * 3
    active = lp = 0
    for k, st in enumerate(steps):
        it = f"{name}: iteration {k + 1}"
        P_sch, P_ev, SOC = AR.homes(cost, hm, *prev, kappa)
        for key, want in (("P_sch", P_sch), ("P_ev", P_ev), ("SOC", SOC)):
            bad = st[key] != want
            assert not bad.any(), (it, key, "(home, step) first / count", _first(bad))
        z = AR.next_target(*prev, kappa)
        for f, R in enumerate(Rz):
            sl = slice(off[f], off[f + 1])
            c = AR.certify_projection(R, z[sl], st["P_est"][sl], u, tol=TOL)
            worst = int(np.argmax(c["resid"]))
            assert c["ok"].all(), (it, f"zone {f} ({sizes[f]} residences)", "columns", np.nonzero(~c["ok"])[0][:8].tolist(),
                                   "worst column", worst, "residual", float(c["resid"][worst]), "rows", int(c["rows"][worst]))
            active += int((c["rows"] > 0).sum())
            lp += c["lp"]
        G, diff = AR.dual_update(prev[2], st["P_est"], st["P_sch"], kappa)
        bad = st["Gamma"] != G
        assert not bad.any(), (it, "Gamma", _first(bad))
        d = st["diff"][k]
        rel = np.abs(d - diff) / np.maximum(diff, 1e-300)
        assert (rel <= 1e-14).all() and np.array_equal(d == 0.0, diff == 0.0), (it, "diff", int(np.argmax(rel)), float(rel.max()))
        comp = st["compact"]
        assert np.array_equal(comp["mask"], _pack(st["P_ev"])), (it, "mask", _first(comp["mask"] != _pack(st["P_ev"])))
        assert np.array_equal(comp["P_sch"], st["P_sch"]) and np.array_equal(comp["diff"], st["diff"]), it
        p_ev, soc = expand_schedule(comp["mask"], T, hm["has_ev"], hm["rating"], hm["capacity"], hm["initial"])
        assert np.array_equal(p_ev, st["P_ev"]) and np.array_equal(soc, st["SOC"]), (it, "expand_schedule")
        assert not (st["P_ev"][~ev] != 0.0).any(), it
        prev = (st["P_est"], st["P_sch"], st["Gamma"])
    return active, lp


@pytest.mark.parametrize("name", CASES)
def test_every_iteration_on_its_own(gpu_lib, name):
    sizes, T, trees, hm, cost, kw, K, opts = _case(name)
    ev = hm["has_ev"].astype(bool)
    counts = np.array(_counts(hm))[ev]
    nwin = (hm["end"] - hm["start"])[ev]
    assert (counts[:, 0] <= nwin).all()                           # every home can meet its target
    if name.startswith("T") or name == "padding":
        assert (counts[:, 1] > 24).any() and (counts[:, 1] <= 24).any() and (counts[:, 0] == 0).any()
    Rz = [O.rmat_from_tree(t.parent, t.r)[np.ix_(t.res_node, t.res_node)] for t in trees]
    steps, graph, stats = _run(gpu_lib, sizes, T, trees, hm, cost, kw, K, opts)
    active, _ = check_steps(name, sizes, Rz, hm, cost, kw, steps)
    assert active > 0                                             # rows bind: certified columns with candidate rows
    assert stats["max_working_set"] >= (17 if name == "handover" else 2), stats["max_working_set"]
    for k, (a, b) in enumerate(zip(steps, graph)):
        for key in ("P_sch", "P_ev", "SOC", "P_est", "Gamma"):
            assert np.array_equal(a[key], b[key]), (name, "captured graph, iteration", k + 1, key)
        assert np.array_equal(a["diff"], b["diff"]), (name, "captured graph, iteration", k + 1, "diff")

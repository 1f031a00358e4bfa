"""The dense operator-QP kernels (utility_qp_warp.cu, utility_qp.cu) on designed columns with a known answer.

Every zone of tests/qp_column_ref.py carries one column per binding-row count m of its sweep (0, 1, 2, 7, 8, 9, ...,
127, 128), so one revs_utility_step call runs the whole range of working-set sizes for that zone: the one-row kernel and
the |W| = 1 Newton path, the warp kernel's admit passes (kAddMaxW), its row cache and the rows read past it (rowp()),
its hand-over at kWW + 1 rows, the CTA classes' pair and register-blocked Hessians, self-verification up to kVerifyMaxN
residences and screening rounds above, up to kWMax rows.  Each zone runs cold, warm from lam*, warm from 1e3 lam*
(g starts low and rises: the verification bound fails on most rows), warm on the wrong rows, without the warp kernel,
with warm sets of up to 16 rows in the warp kernel (REVS_WARP_M_MAX=16) and with the FP64 contraction instead of the
BF16 screen.  Every column must give g* to 1e-8 and lam* to 1e-6 (exactly 0 off the binding rows), pass the KKT check
with the device's multipliers and the solver-independent certificate without them.

Which branch a column takes is asserted where a documented rule decides it: the warm start's support size (the input
of qp_init_kernel's class rule, qp_column_ref.warm_class), cold columns of zones up to kWarpMaxN residences starting in
the warp kernel, and stats()["max_working_set"].  The REVS_DEBUG lines of the host-driven loop give the rest: running
columns per class after each round and the columns the one-row kernel passed on (`fallbacks`).  A warp column handed
to class 1 shows there, because the CTA classes of a round run beside the warp kernel and take it only in the next
round; a CTA column that outgrows its class shows in the next class's count of the same line.  A column the warp
kernel defers (more than kRecheckMaxW rows to recheck) stays in class 0's count and cannot be told from the others."""
import re

import numpy as np
import pytest

import qp_column_ref as Q
from admm_step_ref import certify_projection
from test_gpu_certificates import kkt_check

pytestmark = pytest.mark.gpu

SETTINGS = ["cold", "warm", "warm1e3", "wrong", "nowarp", "mmax16", "screen0"]


def _wrong_rows(zc, seed=5):
    """Warm start on rows that do not bind: in every column, as many rows off A as A has (as far as there are), each
    with the column's mean multiplier.  At m = kWMax the stored rows fill the last class's working set before a single
    binding row is in it: they must leave it first (a solve on W), not end the solve with the overflow error."""
    rng = np.random.default_rng(seed)
    lam0 = np.zeros_like(zc["lam"])
    n = zc["R"].shape[0]
    for t, col in enumerate(zc["cols"]):
        off = np.setdiff1d(np.arange(n), col["A"])
        k = min(len(col["A"]), len(off))
        if k:
            lam0[rng.choice(off, k, replace=False), t] = col["lam"][col["lam"] > 0].mean()
    return lam0


def _lam0(zc, setting):
    if setting in ("warm", "mmax16"):
        return zc["lam"]
    if setting == "warm1e3":
        return 1e3 * zc["lam"]
    if setting == "wrong":
        return _wrong_rows(zc)
    return None


def _run(gpu_lib, zc, setting="cold", lam0=None, repeat=1):
    """[(g, lam)] of `repeat` utility_step calls and the solver's stats, one zone with the dense path forced."""
    tr, n, T = zc["tree"], zc["R"].shape[0], zc["z"].shape[1]
    zero = np.zeros((n, T))
    out = []
    with gpu_lib.Solver([n], T) as s:
        s.set_option("newton_min_n", n)                  # a zone of more than newton_min_n residences takes the tree path
        if setting == "nowarp":
            s.set_option("warp_kernel", 0)
        if setting == "screen0":
            s.set_option("screen", 0)
        s.set_feeder_tree(0, tr.parent, tr.r, tr.res_node)
        for _ in range(repeat):
            out.append(s.utility_step(2.0 * zc["z"], zero, zero, lam0=lam0, **Q.KW))   # target (p_est + p_sch) / 2 = z
        st = s.stats()
    return out, st


def _node_sum(zc, lam):
    """Multipliers with a shared pair's two rows added onto the row that carries lam* of the node."""
    out = lam.copy()
    for t, col in enumerate(zc["cols"]):
        if col["pair"]:
            a, b = col["pair"]
            out[b, t] += out[a, t]
            out[a, t] = 0.0
    return out


def check_columns(zc, g, lam, what):
    """g* to 1e-8, lam* to 1e-6 of the column's largest multiplier and exactly 0 off A, KKT with the device's
    multipliers, the certificate without them."""
    R, z = zc["R"], zc["z"]
    assert np.isfinite(g).all() and np.isfinite(lam).all(), what
    err = np.abs(g - zc["g"]).max(axis=0)
    assert err.max() <= 1e-8, (what, [(m, e) for m, e in zip(zc["ms"], err) if e > 1e-8])
    ls = _node_sum(zc, lam)
    for t, (m, col) in enumerate(zip(zc["ms"], zc["cols"])):
        act = col["lam"] > 0
        on = np.zeros(len(act), bool)
        on[col["A"]] = True
        assert (ls[~on, t] == 0.0).all(), (what, m, "multiplier off the binding rows", np.nonzero(ls[~on, t])[0][:8])
        if act.any():
            e = np.abs(ls[act, t] - col["lam"][act]).max()
            assert e <= 1e-6 * col["lam"].max(), (what, m, e / col["lam"].max())
    kkt_check([R], z, g, lam, Q.U, what)
    cert = certify_projection(R, z, g, Q.U)
    assert cert["ok"].all(), (what, cert["resid"])


# ------------------------------------------------------------------------------------------------ every zone, every start
@pytest.mark.parametrize("setting", SETTINGS)
@pytest.mark.parametrize("name", list(Q.CASES))
def test_designed_columns(gpu_lib, monkeypatch, name, setting):
    zc = Q.case(name)
    n = zc["R"].shape[0]
    ms = zc["ms"]
    if setting == "mmax16":
        monkeypatch.setenv("REVS_WARP_M_MAX", str(Q.C["kWW"]))     # read when the solver is created
    lam0 = _lam0(zc, setting)
    out, st = _run(gpu_lib, zc, setting, lam0, repeat=2 if setting == "cold" else 1)
    g, lam = out[0]
    check_columns(zc, g, lam, (name, setting))
    rows = [m - (1 if c["pair"] else 0) for m, c in zip(ms, zc["cols"])]      # a shared pair binds as one row
    assert st["max_working_set"] >= max(rows), (name, setting, st["max_working_set"])
    if setting == "cold":
        g2, lam2 = out[1]
        assert g.tobytes() == g2.tobytes() and lam.tobytes() == lam2.tobytes(), name
    if setting in ("warm", "mmax16"):
        # the input of qp_init_kernel's rule: the support of the warm start is the binding set, of size m per column
        supp = (lam0 > 0).sum(axis=0)
        assert list(supp) == rows
        wm = Q.C["kWW"] if setting == "mmax16" else None
        classes = {Q.warm_class(n, int(k), wm) for k in supp}
        if supp.max() > Q.CLASS_CAPS[2]:                # the sweep starts columns in every class the zone can use
            assert classes == ({0, 1, 2, 3} if n <= Q.C["kWarpMaxN"] else {1, 2, 3}), (name, classes)


# ------------------------------------------------------------------------------------------------ routing evidence
_LINE = re.compile(r"\[revs\] admm -?\d+ round (\d+): running (\d+) by class (\d+)/(\d+)/(\d+)/(\d+) .*max_ws (\d+) "
                   r".*fallbacks (\d+)")


@pytest.mark.parametrize("name", ["n16", "n128", "n192", "n320", "n513"])
def test_debug_lines_show_each_class(gpu_lib, monkeypatch, capfd, name):
    """Cold start with REVS_DEBUG: every class a column must pass through shows running columns in some round, the
    one-row kernel passes on every column with two or more binding rows (zones up to 128 residences), and the solve
    ends with nothing running."""
    zc = Q.case(name)
    n, ms = zc["R"].shape[0], zc["ms"]
    monkeypatch.setenv("REVS_DEBUG", "1")
    capfd.readouterr()
    out, st = _run(gpu_lib, zc)
    lines = [tuple(int(x) for x in m.groups()) for m in _LINE.finditer(capfd.readouterr().err)]
    check_columns(zc, *out[0], (name, "debug"))
    assert lines, "no REVS_DEBUG round lines"
    assert [ln[0] for ln in lines] == list(range(len(lines)))
    assert lines[-1][1] == 0 and lines[-1][6] >= max(ms), lines[-1]
    seen = [max(ln[2 + c] for ln in lines) for c in range(4)]
    if n <= Q.C["kWarpMaxN"]:
        # cold columns start in the warp kernel; those needing more than kWW rows are handed to class 1 and onwards
        if max(ms) > Q.C["kWW"]:
            assert seen[1] >= 1, lines
    if max(ms) > Q.CLASS_CAPS[1]:
        assert seen[2] >= 1, lines
    if max(ms) > Q.CLASS_CAPS[2]:
        assert seen[3] >= 1, lines
    if n <= 128:
        assert lines[-1][7] >= sum(m >= 2 for m in ms), lines[-1]


# ------------------------------------------------------------------------------------------------ overflow and warm starts
def test_column_beyond_the_last_class_fails(gpu_lib):
    """A column that needs kWMax + 1 binding rows raises RevsError, cold and warm: no projection is returned."""
    tr, R, col = Q.overflow_column()
    n = R.shape[0]
    z = col["z"][:, None]
    zero = np.zeros((n, 1))
    for lam0 in (None, col["lam"][:, None]):
        with gpu_lib.Solver([n], 1) as s:
            s.set_option("newton_min_n", n)
            s.set_feeder_tree(0, tr.parent, tr.r, tr.res_node)
            with pytest.raises(gpu_lib.RevsError):
                s.utility_step(2.0 * z, zero, zero, lam0=lam0, **Q.KW)


def test_warm_start_entries_that_are_not_positive(gpu_lib):
    """lam0 with negative, zero and NaN entries on rows that do not bind: only the positive entries start the working
    set, and every row that does not bind comes back with a zero multiplier."""
    zc = Q.case("n128")
    n, T = zc["R"].shape[0], zc["z"].shape[1]
    rng = np.random.default_rng(4)
    lam0 = zc["lam"].copy()
    for t, col in enumerate(zc["cols"]):
        off = np.setdiff1d(np.arange(n), col["A"])
        if len(off) >= 3:
            a, b, c = rng.choice(off, 3, replace=False)
            lam0[a, t], lam0[b, t], lam0[c, t] = -1.0, -0.0, np.nan
    assert np.isnan(lam0).sum() >= T - 2 and (lam0 < 0).sum() >= T - 2
    out, _ = _run(gpu_lib, zc, "warm", lam0)
    check_columns(zc, *out[0], "lam0 not positive")


def test_warm_start_beyond_the_carried_rows(gpu_lib):
    """A warm start positive on more than kWMax rows of a 300-residence zone: the rows past kWMax are dropped (and
    re-admitted when violated); the result is the designed projection, with no multiplier left off A."""
    zc = Q.zone_case(300, seed=11)
    n = zc["R"].shape[0]
    rng = np.random.default_rng(6)
    lam0 = zc["lam"].copy()
    for t, col in enumerate(zc["cols"]):
        off = np.setdiff1d(np.arange(n), col["A"])
        lam0[rng.choice(off, min(200, len(off)), replace=False), t] = 0.5 * zc["lam"][:, t].max() if col["A"].size else 1.0
    assert ((lam0 > 0).sum(axis=0) > Q.C["kWMax"]).all()
    for setting in ("warm", "nowarp"):
        out, _ = _run(gpu_lib, zc, setting, lam0)
        check_columns(zc, *out[0], ("beyond kWMax", setting))

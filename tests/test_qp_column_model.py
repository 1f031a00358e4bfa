"""The designed columns of tests/qp_column_ref.py (no GPU): each is what it claims to be, and has the answer it claims.

Every case is checked for its shape (exactly m binding rows, strict complementarity margins, band rows inside the BF16
screen's recheck band), for the arithmetic that puts it on a branch of the dense QP kernels (cache rows of the warp
kernel, warm-start class, Hessian variant of the CTA kernels -- from the constants of the CUDA sources), and for its
answer: the oracle's project_voltage finds g* and lam*, and admm_step_ref.certify_projection accepts g* and rejects g*
moved off its face.  test_gpu_qp_shapes.py runs the kernels on the same columns."""
import numpy as np
import pytest

import revs_oracle as O
import qp_column_ref as Q
from admm_step_ref import certify_projection

C = Q.C


# ------------------------------------------------------------------------------------------------ the sweep
def test_sweep_straddles_every_boundary():
    """Each boundary read from the sources has a designed m on both sides of it."""
    ms = set(Q.M_SWEEP)
    edges = [C["kAddMaxW"], C["kWW"], C["kPairM"]] + list(Q.CLASS_CAPS[1:3])
    for e in edges:
        assert {e, e + 1} <= ms, e
    assert C["kWMax"] in ms and 0 in ms and 1 in ms and 2 in ms
    assert Q.WARP_M_MAX in ms and Q.WARP_M_MAX + 1 in ms
    # every change of the CTA kernels' Hessian variant, inside each class's range
    for cls in (1, 2, 3):
        lo = Q.CLASS_CAPS[cls - 1] + 1 if cls > 1 else 1
        for m in range(max(lo, 1), Q.CLASS_CAPS[cls]):
            if Q.hess_variant(m, cls) != Q.hess_variant(m + 1, cls) and m >= 2:
                assert {m, m + 1} <= ms, (cls, m)


def test_sizes_cover_every_zone_class():
    """Zone sizes on both sides of every padding, warp-instantiation, self-verification and path boundary."""
    sizes = set(Q.ZONE_SIZES)
    for e in (128, 192, 256, C["kWarpMaxN"], C["kVerifyMaxN"]):
        assert {e, e + 1} <= sizes, e
    assert {Q.warp_nj(n) for n in sizes} == {4, 6, 8, 10, None}
    assert 2048 in sizes and min(sizes) == 16


def test_uncached_rows_are_reached():
    """For every warp zone whose row cache is smaller than kWW, the sweep has a column with every working row cached
    and one that reads rows past the cache (rowp() from global memory)."""
    reached = 0
    for n in Q.ZONE_SIZES:
        if Q.warp_nj(n) is None:
            continue
        rows = Q.warp_cache_rows(n)
        ms = Q.zone_ms(n)
        if rows >= C["kWW"]:
            assert all(Q.uncached_rows(n, m) == 0 for m in ms), n
            continue
        assert any(m <= rows and m > 1 for m in ms) and any(Q.uncached_rows(n, m) > 0 for m in ms), n
        assert Q.uncached_rows(n, C["kWW"]) == C["kWW"] - rows
        reached += 1
    assert reached >= 5          # zones of 128, 192, 193, 256, 257, 320 residences


def test_warm_classes():
    """qp_init_kernel's rule on the designed sizes: class 0 up to warp_m_max in warp zones, then by the class caps."""
    assert Q.warm_class(128, Q.WARP_M_MAX) == 0 and Q.warm_class(128, Q.WARP_M_MAX + 1) == 1
    assert Q.warm_class(320, C["kWW"], warp_m_max=C["kWW"]) == 0
    assert Q.warm_class(321, 0) == 1
    for cls in (1, 2, 3):
        assert Q.warm_class(513, Q.CLASS_CAPS[cls]) == cls
        if cls < 3:
            assert Q.warm_class(513, Q.CLASS_CAPS[cls] + 1) == cls + 1
    assert Q.warm_class(2048, 300) == 3


# ------------------------------------------------------------------------------------------------ the columns
def _check_shape(name, zc):
    R, u = zc["R"], Q.U
    n = R.shape[0]
    assert zc["ms"] == [m for m in Q.zone_ms(n) if m <= n - 2 * max(len(zc["pairs"]) - 1, 0)]
    for t, (m, col) in enumerate(zip(zc["ms"], zc["cols"])):
        g, lam, z = col["g"], col["lam"], col["z"]
        v = R @ g
        A = col["A"]
        off = np.ones(n, bool)
        off[A] = False
        what = (name, t, m)
        assert len(A) == m and len(np.unique(A)) == m, what
        node_rows = m - (1 if col["pair"] else 0)                     # one multiplier per node
        assert (lam > 0).sum() == node_rows and (lam[off] == 0).all(), what
        if m:
            assert np.abs(v[A] - u).max() <= 1e-13 * u, what
            assert g[A].min() > 0.0, what
        if off.any():
            assert v[off].max() <= u * (1.0 - Q.SLACK), what
        assert g.min() >= 0.0 and (g[col["Z"]] == 0.0).all(), what
        w = z - R @ lam
        F = g > 0
        assert np.abs(g[F] - w[F]).max() <= 1e-12 * max(1.0, np.abs(z).max()), what
        if len(col["Z"]):
            assert w[col["Z"]].max() < 0.0, what                       # strictly below zero: a margin on the g = 0 side
        B = col["band"]
        if len(B):
            assert ((v[B] > (1.0 - Q.SCREEN_MARGIN) * u) & (v[B] < u)).all(), what
        if col["pair"]:
            a, b = col["pair"]
            assert np.array_equal(R[a], R[b]) and a in A and b in A, what


@pytest.mark.parametrize("name", list(Q.CASES))
def test_designed_columns_are_what_they_claim(name):
    zc = Q.case(name)
    _check_shape(name, zc)
    spec = Q.CASES[name]
    if spec.get("band"):
        n = spec["n"]
        assert all(len(c["band"]) == min(spec["band"], max(n - len(c["A"]) - 1, 0)) for c in zc["cols"]), name
    if spec.get("shared"):
        assert sum(c["pair"] is not None for c in zc["cols"]) >= 10, name
        assert any(c["pair"] is not None and len(c["A"]) >= 64 for c in zc["cols"]), name


@pytest.mark.parametrize("name", list(Q.CASES))
def test_oracle_finds_the_designed_projection(name):
    """The oracle's project_voltage returns g* to 1e-8 and, per node, lam* to 1e-6 relative."""
    zc = Q.case(name)
    R = zc["R"]
    for t, (m, col) in enumerate(zip(zc["ms"], zc["cols"])):
        g, lam, _ = O.project_voltage(col["z"], R, Q.U)
        assert np.abs(g - col["g"]).max() <= 1e-8, (name, t, m, np.abs(g - col["g"]).max())
        ls = lam.copy()
        if col["pair"]:
            a, b = col["pair"]
            ls[b] += ls[a]
            ls[a] = 0.0
        act = col["lam"] > 0
        if act.any():
            assert np.abs(ls[act] - col["lam"][act]).max() <= 1e-6 * col["lam"].max(), (name, t, m)
        assert np.abs(ls[~act]).max(initial=0.0) <= 1e-9 * max(col["lam"].max(), 1.0), (name, t, m)


@pytest.mark.parametrize("name", ["n128", "n320", "n513", "band320", "shared300"])
def test_certificate_accepts_the_solution_and_rejects_a_moved_one(name):
    zc = Q.case(name)
    R, z, g = zc["R"], zc["z"], zc["g"]
    cert = certify_projection(R, z, g, Q.U)
    assert cert["ok"].all(), (name, cert["resid"])
    assert np.array_equal(cert["rows"], [len(c["A"]) for c in zc["cols"]])
    # off the face: the binding homes lowered by 1e-6 of their value (still feasible, no longer optimal)
    moved = g.copy()
    for t, col in enumerate(zc["cols"]):
        sel = col["A"] if len(col["A"]) else np.nonzero(g[:, t] > 0)[0]
        moved[sel, t] *= 1.0 - 1e-6
    bad = certify_projection(R, z, moved, Q.U)
    assert not bad["ok"].any(), (name, bad["ok"])


def test_overflow_column_needs_more_rows_than_the_last_class():
    tr, R, col = Q.overflow_column()
    assert len(col["A"]) == C["kWMax"] + 1 == (col["lam"] > 0).sum()
    g, _, _ = O.project_voltage(col["z"], R, Q.U)
    assert np.abs(g - col["g"]).max() <= 1e-8

"""The BF16 voltage screen at its worst case, and the verification bound the warp QP kernels build on it.

The screen computes v~ = R~ g~ (BF16 operands, FP32 accumulation on the tensor cores).  Its result is used twice:
rows with v~ <= (1 - kScreenMargin) u are taken as feasible, and the warp QP kernels store kScreenUp * v~ as an
upper bound of the row's true voltage, which proves rows feasible after a solve without an exact recheck.  Both
rest on  v <= kScreenUp * v~  for every non-negative R, g and every K up to kScreenMaxN.

Worst case: an operand whose significand sits just below a BF16 rounding midpoint loses 2^-8 of its value, so a
product of two loses ~2^-7 (v / v~ = 1.0078) before any accumulation error.
"""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "revs-admm_b200", "csrc")


def _constant(fname, name):
    with open(os.path.join(CSRC, fname)) as f:
        m = re.search(r"constexpr\s+(?:double|int)\s+%s\s*=\s*([0-9.eE+-]+)\s*;" % name, f.read())
    assert m, f"{name} not found in {fname}"
    return float(m.group(1))


SCREEN_UP = _constant("common.cuh", "kScreenUp")
SCREEN_MARGIN = _constant("common.cuh", "kScreenMargin")
SCREEN_MAX_N = int(_constant("common.cuh", "kScreenMaxN"))
# FP32 accumulation of the tensor cores, measured on a B200 for both kernels (profiles/exp_screen_accumulation.py,
# profiles/exp_screen_accumulation_b200.json): never above the exact sum of the products, and 1 + n small terms comes
# out as 1 + floor(their sum) in ulps of 1 -- a truncating accumulator, so up to one ulp (2 * 2^-24 relative) per step.
C_ACC = 2
U24 = 2.0 ** -24
W = 1.0 + 2.0 ** -8 - 2.0 ** -20          # just below the midpoint of [1, 1 + 2^-7]: rounds down to 1, exact in FP32


def bf16(x):
    """__float2bfloat16_rn((float)x) of every element, as float64 (finite inputs)."""
    b = np.ascontiguousarray(x, dtype=np.float64).astype(np.float32).view(np.uint32)
    b = (b + np.uint32(0x7FFF) + ((b >> np.uint32(16)) & np.uint32(1))) & np.uint32(0xFFFF0000)
    return b.view(np.float32).astype(np.float64)


def exact_bf16_product(A, B):
    """Exact sum of the BF16-rounded products (A~ B~): the operands scaled to integers, every partial sum of the FP64
    product is then an integer below 2^53."""
    Ab, Bb = bf16(A), bf16(B)

    def scale(X):
        nz = X[X > 0]
        e = int(np.floor(np.log2(nz.min()))) - 7 if nz.size else 0       # BF16: 8 significant bits
        return X * 2.0 ** -e, e

    Ai, ea = scale(Ab)
    Bi, eb = scale(Bb)
    assert np.array_equal(Ai, np.round(Ai)) and np.array_equal(Bi, np.round(Bi))
    assert Ai.max() * Bi.max() * A.shape[1] < 2.0 ** 53, "operands too spread for an exact integer sum"
    return (Ai @ Bi) * 2.0 ** (ea + eb)


# ----------------------------------------------------------------- the constants (no GPU)
def test_screen_constants_cover_the_worst_case():
    """kScreenUp covers two operands rounded by 2^-8 each (the FP64 -> FP32 -> BF16 double rounding included) and
    C_ACC K 2^-24 of accumulation at K = kScreenMaxN; rows below the candidate threshold stay provably feasible."""
    with open(os.path.join(CSRC, "revs_capi.cu")) as f:
        capi = f.read()
    assert "16384" not in capi and capi.count("kScreenMaxN") >= 2       # both places the limit is enforced use it
    worst = 1.0 / ((1.0 - 2.0 ** -8) ** 2 * (1.0 - C_ACC * SCREEN_MAX_N * U24))
    assert SCREEN_UP >= worst, (SCREEN_UP, worst)
    assert (1.0 - SCREEN_MARGIN) * SCREEN_UP < 1.0
    # the worst-case operand of the tests below really loses 2^-8: x / bf16(x) just below 1 + 2^-8
    assert bf16(np.array([W]))[0] == 1.0 and W / 1.0 > 1.0 + 2.0 ** -8 - 2.0 ** -19


def test_bf16_emulation_matches_torch():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(3)
    x = np.concatenate([rng.uniform(0, 10, 20000), np.exp2(rng.uniform(-30, 30, 20000)), [0.0, 1.0, W, 2 * W],
                        (1.0 + (np.arange(256) + 0.5) * 2.0 ** -7) * 2.0 ** -3])          # exact midpoints: ties to even
    x = np.concatenate([x, -x])
    ref = torch.from_numpy(x).to(torch.float32).to(torch.bfloat16).to(torch.float64).numpy()
    assert np.array_equal(bf16(x), ref)


# ----------------------------------------------------------------- worst-case operands through the kernels
def _worst_operands(M, K, T, mixed, seed):
    """Non-negative A (M x K), B (K x T): entries W * 2^e (lose 2^-8 to BF16), with power-of-two scales in the range of
    R and g; `mixed` also draws exact BF16 values and zeros."""
    rng = np.random.default_rng(seed)
    A = W * np.exp2(rng.integers(-12, -6, (M, K)).astype(float))
    B = W * np.exp2(rng.integers(-3, 3, (K, T)).astype(float))
    if mixed:
        for X in (A, B):
            pick = rng.random(X.shape)
            X[pick < 0.3] = bf16(X[pick < 0.3] * rng.uniform(0.5, 1.0, int((pick < 0.3).sum())))
            X[pick > 0.8] = 0.0
    return A, B


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 5, 95, 96, 97, 100, 256])
@pytest.mark.parametrize("K", [1, 15, 16, 17, 64, 1008, 4096, 16384])
def test_screen_worst_case_operands(gpu_lib, K, T):
    impls = [0, 1] if T <= 96 else [0]            # the tcgen05 kernel takes T <= 96, the solver uses impl 0 above
    for mixed in (False, True):
        A, B = _worst_operands(300, K, T, mixed, seed=K * 1000 + T)
        for M in (1, 127, 128, 129, 300):
            a = A[:M]
            ref_a = a @ B                                  # the FP64 product of the inputs
            ref_b = exact_bf16_product(a, B)               # exact sum of the BF16-rounded products
            acc = C_ACC * K * U24 * ref_b
            C = {impl: gpu_lib.screen_contract(a, B, impl=impl) for impl in impls}
            for impl, c in C.items():
                what = (impl, M, K, T, mixed)
                assert (ref_a <= SCREEN_UP * c).all(), (what, (ref_a / np.where(c > 0, c, 1.0)).max())
                assert (np.abs(c - ref_b) <= acc).all(), (what, (np.abs(c - ref_b) / np.maximum(acc, 1e-300)).max())
            if len(C) == 2:
                assert (np.abs(C[0] - C[1]) <= acc).all(), (M, K, T, mixed)
            if not mixed:                                  # every product loses (1 + 2^-8)^2 to the rounding
                assert (ref_a > 1.0078 * C[0]).all(), (M, K, T)


# ----------------------------------------------------------------- realistic zones
@pytest.mark.gpu
@pytest.mark.parametrize("name,feeders", [("refshape", 6), ("laterals", 3)])
def test_screen_bound_on_population_zones(gpu_lib, name, feeders):
    """R blocks of the benchmark populations against schedules of the oracle's ADMM history (P_est and P_sch)."""
    import revs_oracle as O
    from revs_admm_b200.feeder import population
    trees, hm, cost, sizes, T = population(name, feeders, seed=0)
    Rb = [t.rmat()[np.ix_(t.res_node, t.res_node)] for t in trees]
    hist = O.solve_ADMM_arrays(Rb, load=hm["load"], cost=cost, ev_mask=hm["has_ev"].astype(bool), rating=hm["rating"],
                               capacity=hm["capacity"], initial=hm["initial"], start=hm["start"], end=hm["end"],
                               kappa=5.0, iter_max=6, vset=1.03, vlow=0.95, vhigh=1.05, return_history=True)["history"]
    G = np.concatenate([hist[k][j] for k in (0, 2, 5) for j in (0, 1)], axis=1)      # [H, 6 T] non-negative schedules
    assert G.min() >= 0.0
    worst, rows = 0.0, 0
    off = 0
    for R in Rb:
        n = R.shape[0]
        g = G[off:off + n]
        off += n
        ref = R @ g
        for impl in (0, 1):
            for t0 in range(0, g.shape[1], 96):
                c = gpu_lib.screen_contract(R, g[:, t0:t0 + 96], impl=impl)
                r = ref[:, t0:t0 + 96]
                assert (r <= SCREEN_UP * c).all(), (name, impl, (r / np.where(c > 0, c, 1.0)).max())
                pos = c > 0
                if pos.any():
                    worst = max(worst, float((r[pos] / c[pos]).max()))
                    rows += int(pos.sum())
    print(f"{name}: largest v / v~ over {rows} (row, step) pairs: {worst:.6f}")
    assert worst > 1.0


# ----------------------------------------------------------------- end to end: the warp kernels' verification bound
KQP_TOL = 1e-11             # csrc/revs_capi.cu kQpTol


def kkt_check(Rblocks, z, g, lam, u, what=""):
    """Assert the KKT conditions zone by zone (same check as test_gpu_certificates.py); returns the largest multiplier
    and the number of active rows."""
    off, worst_lam, n_active = 0, 0.0, 0
    for R in Rblocks:
        n = R.shape[0]
        sl = slice(off, off + n)
        gz, lz, zz = g[sl], lam[sl], z[sl]
        v = R @ gz
        assert gz.min() >= 0.0, what
        assert (v - u).max() <= 1e-9, (what, (v - u).max())
        assert lz.min() >= 0.0, what
        stat = np.abs(gz - np.maximum(zz - R @ lz, 0.0)).max()
        assert stat <= 1e-9, (what, stat)
        act = lz > 0
        if act.any():
            assert np.abs(v[act] - u).max() <= 1e-9, (what, np.abs(v[act] - u).max())
            worst_lam = max(worst_lam, lz.max())
            n_active += int(act.sum())
        off += n
    return worst_lam, n_active


def _verification_case(two_rows, n=32, vset=1.03, vhigh=1.05):
    """One zone, one column, on which a verification bound below the true screening ratio accepts a violated row.

    Row B has every entry w = W 2^-7 (BF16: 2^-7); the loads' g = W 2^f (BF16: 2^f), so v_B = W^2 v~_B exactly, with
    v~_B just below the candidate threshold 0.99 u: B is not rechecked, its bound is factor * v~_B.  Row A1 has entries
    about w on the loads (one of them half of it), tuned so that at the optimum of the rows A1 (and A2) alone, v_A1 = u
    and v_B slightly exceeds u.  The warm start lam0 on A1 (and A2: half the loads, entries c / 2) is too large: the
    solve lowers it, g rises by D+, and the verification bound of B, factor * v~_B + w D+, stays below u for every
    factor up to `accept` although B is violated.  Homes A1, A2, B have z < 0 (g = 0).  No two rows are proportional
    on the loads, so the working-set Hessians stay regular.
    """
    u = vhigh ** 2 - vset ** 2
    thr = (1.0 - SCREEN_MARGIN) * u
    a1, a2, b = 0, (1 if two_rows else None), (2 if two_rows else 1)
    loads = np.arange(3 if two_rows else 2, n)
    w = W * 2.0 ** -7
    # g~ of the loads: powers of two summing to just below thr / 2^-7 (exact in FP32)
    target = thr * 2.0 ** 7 * (1.0 - 1e-4)
    f = np.full(len(loads), -3)
    for i in range(len(loads)):
        while np.exp2(f).sum() + 2.0 ** f[i] <= target and f[i] < 0:
            f[i] += 1
    g_old = W * np.exp2(f.astype(float))
    vt_b = 2.0 ** -7 * np.exp2(f.astype(float)).sum()
    goal = u + 0.5 * (W * W - 1.005) * vt_b                    # v_B at the optimum: inside the window

    def build(c):
        c = float(np.float32(c))                               # short significand: R lam0 and z - R lam0 are exact
        R = np.zeros((n, n))
        R[loads, loads] = w / 8
        R[b, :] = R[:, b] = w
        R[a1, loads] = R[loads, a1] = c
        R[a1, loads[-1]] = R[loads[-1], a1] = c / 2
        R[a1, a1] = c
        lam0 = np.zeros(n)
        lam0[a1] = 1.0
        if two_rows:
            half = loads[: len(loads) // 2]
            R[a2, half] = R[half, a2] = c / 2
            R[a2, a2], R[a1, a2], R[a2, a1] = c, c / 2, c / 2
            lam0[a2] = 0.25
        z = np.full(n, -1.0)
        z[loads] = g_old + R[loads] @ lam0
        r1 = R[a1, loads]
        lam_a1 = (r1 @ z[loads] - u) / (r1 @ r1)               # v_A1 = u with every load positive, lam_A2 = 0
        g_new = np.maximum(z - R[:, a1] * lam_a1, 0.0)
        return R, z, lam0, lam_a1, g_new

    lo, hi = 0.95 * w, 1.05 * w                                # v_B at the optimum falls as A1 gets heavier
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if w * build(mid)[4].sum() > goal else (lo, mid)
    R, z, lam0, lam_a1, g_new = build(hi)
    g_init = np.maximum(z - R @ lam0, 0.0)                     # what qp_init_kernel writes
    assert np.array_equal(g_init[loads], g_old)
    assert np.array_equal(bf16(R[b]), np.full(n, 2.0 ** -7)) and np.array_equal(bf16(g_old), np.exp2(f.astype(float)))
    v_old = R @ g_init
    assert thr * 0.985 < vt_b <= thr                                           # B is no candidate
    assert v_old[b] == pytest.approx(W * W * vt_b, rel=1e-15)
    assert v_old[a1] < u                                                       # lam0 is too large on A1
    assert lam_a1 > 0 and (g_new[loads] > 0).all() and abs(R[a1] @ g_new - u) <= 1e-12
    if two_rows:
        assert R[a2] @ g_new < u
    dplus = np.maximum(g_new - g_init, 0.0).sum()
    v_b_new = R[b] @ g_new
    accept = (u + KQP_TOL - R[b].max() * dplus * (1.0 + 1e-9)) / vt_b   # largest factor that passes row B unchecked
    assert v_b_new > u + 1e-6                                            # B is violated at that point
    assert 1.005 < accept < W * W                                        # a factor under the true ratio accepts it
    return dict(R=R, z=z, lam0=lam0, u=u, vset=vset, vhigh=vhigh, b=b)


@pytest.mark.gpu
@pytest.mark.parametrize("impl", [0, 1])
@pytest.mark.parametrize("two_rows", [False, True], ids=["one_row_kernel", "general_warp_kernel"])
def test_verification_bound_keeps_worst_case_row(gpu_lib, two_rows, impl):
    """A warm start with one (two) too-large multiplier(s) goes to utility_qp_fast_kernel (utility_qp_warp_kernel<4>);
    row B, screened at its worst-case ratio, must not be accepted by the verification bound."""
    case = _verification_case(two_rows)
    R, n, T = case["R"], case["R"].shape[0], 4
    Z = np.repeat(case["z"][:, None], T, axis=1)
    zero = np.zeros((n, T))
    with gpu_lib.Solver([n], T) as s:
        s.set_sensitivity(0, R)
        s.set_option("screen_impl", impl)
        g, lam = s.utility_step(2.0 * Z, zero, zero, kappa=5.0, vset=case["vset"], vlow=0.95, vhigh=case["vhigh"],
                                lam0=np.repeat(case["lam0"][:, None], T, axis=1))
    for t in range(T):
        kkt_check([R], Z[:, t], g[:, t], lam[:, t], case["u"], f"step {t}")
    assert (lam[case["b"]] > 0).all()                 # the worst-case row binds

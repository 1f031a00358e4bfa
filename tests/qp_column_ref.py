"""Designed operator-QP columns with a known answer (numpy, no GPU), for the dense QP kernels' shape tests.

A column is built backwards from its solution.  In a zone with sensitivity block R (positive definite: every residence
has its own service line, so rows of distinct residences are linearly independent):
    pick a binding set A of exactly m residences, homes Z outside A held at zero, draws g*_N > 0 on the rest;
    solve R_AA g*_A = u - R_{A,.} g*_{not A} in fp64, and redraw until g*_A clears a floor and every row off A is at
    most u (1 - kSlack);
    pick multipliers lam*_A > 0 and set z = g* + R_{.A} lam* where g* > 0, z_j = (R lam*)_j - delta_j on Z.
Then g* = [z - R lam*]_+, R g* <= u with equality exactly on A, lam* > 0 exactly on A: the KKT conditions of
min 1/2 |g - z|^2 s.t. g >= 0, R g <= u hold, so g* is the projection and lam* its unique multiplier -- exact up to
rounding, whatever a solver does.

Variants: `band` rows of N placed inside the BF16 screen's recheck band (1 - kScreenMargin) u < v < u (1 - kSlack),
solved for together with A; a zone with `shared` pairs of residences on one node (identical rows: lam is not unique,
g is; a pair binds together); m = 0 (g = [z]_+).

The kernels' branch boundaries are read from the CUDA sources, so that a change of a cache size or a class cap moves
the designed cases with it."""
import os
import re

import numpy as np

import revs_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "revs-admm_b200", "csrc")

U = 1.05 ** 2 - 1.03 ** 2          # vhigh^2 - vset^2 of the tests (vset 1.03, vhigh 1.05)
KW = dict(kappa=5.0, vset=1.03, vlow=0.95, vhigh=1.05)
SLACK = 1e-3                       # rows off A stay at most u (1 - SLACK)
FLOOR = 1e-2                       # g*_A >= FLOOR * (median of g*_N): binding homes carry load


def _source(fname):
    with open(os.path.join(CSRC, fname)) as f:
        return f.read()


def constant(fname, name):
    """Value of `constexpr int|double name = <literal>;` or `#define name <literal>` in a CUDA source."""
    src = _source(fname)
    m = re.search(r"constexpr\s+(?:double|int)\s+%s\s*=\s*([0-9.eE+-]+)\s*;" % name, src)
    if not m:
        m = re.search(r"#define\s+%s\s+([0-9.eE+-]+)\b" % name, src)
    assert m, f"{name} not found in {fname}"
    return float(m.group(1))


def _class_caps():
    """qp_class_cap(0..3) of common.cuh: kWW, then the literals of classes 1 and 2, then kWMax."""
    m = re.search(r"qp_class_cap\(int cls\)\s*\{\s*return\s+cls == 0 \? (\w+) : \(cls == 1 \? (\w+) : "
                  r"\(cls == 2 \? (\w+) : (\w+)\)\);", _source("common.cuh"))
    assert m, "qp_class_cap not found in common.cuh"
    return tuple(int(C[v]) if v in C else int(v) for v in m.groups())


C = {k: int(constant("common.cuh", k)) for k in ("kWW", "kWMax", "kPad", "kVerifyMaxN", "kWarpMaxN")}
C.update({k: int(constant("utility_qp_warp.cu", k)) for k in
          ("kAddMaxW", "kHysteresisW", "kCacheDoubles", "REVS_WARP_CACHE_BIG", "kRecheckMaxW")})
C["kPairM"] = int(constant("utility_qp.cu", "kPairM"))
C["kChgMax"] = int(constant("utility_qp.cu", "kChgMax"))
SCREEN_MARGIN = constant("common.cuh", "kScreenMargin")
CLASS_CAPS = _class_caps()
WARP_M_MAX = C["kWW"] - C["kHysteresisW"]          # default warm-start threshold of class 0 (qp_warp_m_max_default)


# ------------------------------------------------------------------------------------------------ branch arithmetic
def padded(n):
    """Leading dimension n_p of the zone's R block: n rounded up to a multiple of kPad."""
    return -(-n // C["kPad"]) * C["kPad"]


def warp_nj(n):
    """Homes per lane of the warp kernel that runs a zone of n residences alone in its solver (None: no warp kernel)."""
    if n > C["kWarpMaxN"]:
        return None
    if n <= 128:
        return 4
    return 6 if n <= 192 else (8 if n <= 256 else 10)


def warp_cache_rows(n):
    """Working rows of R the warp kernel keeps in shared memory for a zone of n residences (kCache / ld)."""
    nj = warp_nj(n)
    cache = C["kCacheDoubles"] if nj == 4 else C["REVS_WARP_CACHE_BIG"]
    return cache // padded(n)


def uncached_rows(n, m):
    """Working rows the warp kernel reads from global memory (rowp() past the cache) at |W| = m."""
    if warp_nj(n) is None or m > C["kWW"]:
        return 0
    return max(0, m - min(m, warp_cache_rows(n)))


def warm_class(n, m, warp_m_max=None):
    """Class qp_init_kernel gives a column whose warm start has m positive multipliers (m <= kWMax carried)."""
    wm = WARP_M_MAX if warp_m_max is None else warp_m_max
    m = min(m, C["kWMax"])
    cl = 0 if (n <= C["kWarpMaxN"] and m <= wm) else 1
    while cl < len(CLASS_CAPS) - 1 and m > CLASS_CAPS[cl]:
        cl += 1
    return cl


def hess_variant(m, cls):
    """(kind, NP, NQ) of the model Hessian the CTA kernel of class cls forms at |W| = m (utility_qp.cu)."""
    if m <= C["kPairM"]:
        return ("pairs", 0, 0)
    threads = 128 if cls == 1 else 256
    ty = threads // 16
    nq, np_ = (m + 15) >> 4, (m + ty - 1) // ty
    wmax = CLASS_CAPS[cls]
    if wmax == 32:
        return ("hess",) + ((1, 1) if np_ <= 1 else (2, 1) if np_ <= 2 else (3, 2) if np_ <= 3 else (4, 2))
    if nq <= 1:
        return ("hess", 1, 1)
    if nq <= 2:
        return ("hess", 2, 2)
    if nq <= 3:
        return ("hess", 3, 3)
    if nq <= 4 or wmax == 64:
        return ("hess", 4, 4)
    if nq <= 6:
        return ("hess", 6, 6)
    return ("hess", 8, 8)


# ------------------------------------------------------------------------------------------------ zones
def zone(n, seed=0, shared=0):
    """(tree, R) of a synthetic_feeder zone of n residences; `shared` pairs of residences moved onto one node (the
    second residence of a pair takes the first one's node).  Returns also the list of pairs."""
    from revs_admm_b200.feeder import FeederTree, synthetic_feeder
    tr = synthetic_feeder(n, seed=seed)
    # service lines of 1e-2 with a narrow spread: the smallest eigenvalue of R_AA stays near 1e-2, so the kernels' KKT
    # tolerance (1e-11 on the rows) bounds |g - g*| by ~1e-9 even when every home binds
    nx = len(tr.parent) - n
    r = tr.r.copy()
    r[nx:] = 1e-2 * np.random.default_rng(seed).lognormal(0.0, 0.4, n)
    tr = FeederTree(parent=tr.parent, r=r, res_node=tr.res_node, edge_sign=tr.edge_sign)
    pairs = []
    if shared:
        res = tr.res_node.copy()
        step = n // (shared + 1)
        for k in range(shared):
            a = step * (k + 1) - 1
            res[a + 1] = res[a]
            pairs.append((a, a + 1))
        tr = FeederTree(parent=tr.parent, r=tr.r, res_node=res, edge_sign=tr.edge_sign)
    R = O.rmat_from_tree(tr.parent, tr.r)[np.ix_(tr.res_node, tr.res_node)]
    return tr, R, pairs


# ------------------------------------------------------------------------------------------------ columns
def design_column(R, m, rng, u=U, band=0, pairs=(), zero_share=0.15, tries=50):
    """One column with exactly m binding rows.  `band` rows of N are placed at (1 - kScreenMargin) u < v < u (1 - SLACK);
    with `pairs`, the first pair (a, b) of residences on one node binds (both in A, a and b count towards m).

    Returns dict(z, g, lam, A (sorted binding rows), Z (homes held at zero), band (rows in the band), pair (the binding
    pair or None)) where lam is lam* (on a shared pair: all of the node's multiplier on its second residence)."""
    n = R.shape[0]
    d = np.diag(R)
    assert 0 <= m <= n
    # binding homes are drawn among those whose own service line carries most of their row (largest d - max off-diagonal):
    # many binding homes behind one long shared primary path would push the rows between them over u
    own = np.argsort(-(d - (R - np.diag(d)).max(axis=1)) / d, kind="stable")
    npool = min(n, max(2 * m, n // 3))
    for _ in range(tries):
        idx = np.r_[rng.permutation(own[:npool]), rng.permutation(own[npool:])].astype(int)
        pair = pairs[0] if pairs and m >= 2 else None
        paired = {j for p in pairs for j in p}
        free_homes = [i for i in idx if i not in paired]
        first = (list(pair) if pair else []) + free_homes
        assert m <= len(first), "a shared node other than the binding pair would bind too"
        A = np.array(first[:m], dtype=int)
        rest = np.array(first[m:] + [j for j in idx if j in paired and not (pair and j in pair)], dtype=int)
        nb = min(band, max(len(rest) - 1, 0))
        B = rest[:nb]
        Zn = int(zero_share * (len(rest) - nb))
        Zs = rest[nb:nb + Zn]
        N = rest[nb + Zn:]
        g = np.zeros(n)
        g[N] = rng.uniform(0.2, 1.0, len(N))
        if len(N):
            g[N] *= 0.3 * u / max((R[:, N] @ g[N]).max(), 1e-300)
        # solve for the binding rows (and the band rows) on their targets; the second home of a shared pair is drawn
        S = np.r_[A[1:] if pair else A, B].astype(int)
        if pair:
            g[A[0]] = 0.3 * u / (2.0 * d[A[0]]) * rng.uniform(0.5, 1.0)
        tgt = np.r_[np.full(len(S) - len(B), u), u * rng.uniform(1.0 - 0.8 * SCREEN_MARGIN, 1.0 - 2 * SLACK, len(B))]
        free = np.setdiff1d(np.arange(n), S)
        if len(S):
            g[S] = np.linalg.solve(R[np.ix_(S, S)], tgt - R[np.ix_(S, free)] @ g[free])
        med = np.median(g[N]) if len(N) else 1.0
        if len(S) and g[S].min() < FLOOR * med:
            continue
        if pair and g[A[0]] < FLOOR * med:
            continue
        v = R @ g
        off = np.ones(n, bool)
        off[A] = False
        if off.any() and v[off].max() > u * (1.0 - SLACK):
            continue
        if m and np.abs(v[A] - u).max() > 1e-13 * u:
            continue
        if nb and not ((v[B] > (1.0 - SCREEN_MARGIN) * u).all() and (v[B] < u * (1.0 - SLACK)).all()):
            continue
        lam = np.zeros(n)
        act = np.sort(A)
        if pair:
            act = np.sort(np.r_[A[1:]])       # one multiplier per node: on the pair's second home (a row of A)
        lam[act] = rng.uniform(0.3, 1.0, len(act)) * g[act] / d[act]
        rl = R @ lam
        z = g + rl
        delta = rng.uniform(0.05, 0.5, len(Zs)) * med
        z[Zs] = rl[Zs] - delta
        return dict(z=z, g=g, lam=lam, A=np.sort(A), Z=np.sort(Zs), band=np.sort(B), pair=pair)
    raise AssertionError(f"no valid column with m = {m} in {tries} draws")


M_SWEEP = (0, 1, 2, 7, 8, 9, 10, 13, 14, 16, 17, 24, 25, 32, 33, 48, 49, 64, 65, 96, 97, 127, 128)
ZONE_SIZES = (16, 128, 129, 192, 193, 256, 257, 320, 321, 512, 513, 2048)


def zone_ms(n):
    """Binding-row counts of the columns of a zone of n residences: column t carries m_t."""
    return [m for m in M_SWEEP if m <= min(n, C["kWMax"])]


def zone_case(n, seed=None, band=0, shared=0):
    """A zone of n residences and its columns (one per m of zone_ms(n)): dict(tree, R, pairs, ms, z, g, lam [n, T],
    cols (design_column of every column))."""
    seed = n if seed is None else seed
    tr, R, pairs = zone(n, seed=seed, shared=shared)
    rng = np.random.default_rng(1000 + seed)
    ms = [m for m in zone_ms(n) if m <= n - 2 * max(len(pairs) - 1, 0)]
    cols = [design_column(R, m, rng, band=band, pairs=pairs) for m in ms]
    return dict(tree=tr, R=R, pairs=pairs, ms=ms, cols=cols, z=np.stack([c["z"] for c in cols], axis=1),
                g=np.stack([c["g"] for c in cols], axis=1), lam=np.stack([c["lam"] for c in cols], axis=1))


# every designed zone of the shape tests: plain zones at every size class, band rows, shared nodes
CASES = {**{f"n{n}": dict(n=n) for n in ZONE_SIZES},
         "band128": dict(n=128, band=24, seed=7), "band320": dict(n=320, band=24, seed=8),
         "shared128": dict(n=128, shared=3, seed=9), "shared300": dict(n=300, shared=2, band=8, seed=10)}
_cache = {}


def case(name):
    """zone_case of a named zone (memoised: the GPU tests run every zone under several settings)."""
    if name not in _cache:
        kw = dict(CASES[name])
        _cache[name] = zone_case(kw.pop("n"), **kw)
    return _cache[name]


def overflow_column(n=192, seed=3):
    """A zone and one column that needs kWMax + 1 binding rows."""
    tr, R, _ = zone(n, seed=seed)
    col = design_column(R, C["kWMax"] + 1, np.random.default_rng(seed))
    return tr, R, col

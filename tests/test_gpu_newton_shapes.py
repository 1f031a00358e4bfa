"""The tree-Newton operator kernel (csrc/tree_newton.cu) on trees whose shape takes every branch of its data layout.

The kernel walks a zone level by level, one CTA of kNtThreads = 256 threads per column.  Its layout changes with the
shape of the tree:
    a level wider than 256 nodes      a thread handles a second node of the level, whose inputs are loaded in place
                                      (the first one's are prefetched a level ahead)
    a level wider than kXCap = 512    messages to parents and children beyond position 512 go through global memory
                                      instead of the shared-memory exchange (products, tree_solve up and down)
    more than kLvlCap = 1024 levels   level offsets are read from global memory
    several residences on one node    one row and one multiplier per node (shared nodes, contracted edges): the
                                      multiplier goes to the node's first home, a warm start is summed over its homes
    many roots                        a wide level 0; a row with nothing of the piece below and no parent to pin
                                      sits the guess out
The feeders of the rest of the suite stay below all of the first three (172 nodes on the widest level, 141 levels).
Every builder here is asserted, on the host model of newton_build_zone (tests/tree_newton_ref.LevelTree, same 1e-10
contraction), to have the layout it exists for, so that a change to a generator cannot silently drop the coverage.

Each projection returned by revs_utility_step is proved by the KKT conditions with the device's multipliers
(test_gpu_certificates.kkt_check), compared with the dense oracle (or, for the forest, with an exact closed form), and
checked for multiplier placement, warm starts, determinism and independence from the other zones of the solver."""
import numpy as np
import pytest

import revs_oracle as O
from test_gpu_certificates import kkt_check
from tree_newton_ref import LevelTree

U = 1.05 ** 2 - 1.03 ** 2
KW = dict(kappa=5.0, vset=1.03, vlow=0.95, vhigh=1.05)


def _tree(parent, r, res_node):
    from revs_admm_b200.feeder import FeederTree
    parent = np.asarray(parent, dtype=np.int32)
    assert (parent < np.arange(len(parent))).all()
    return FeederTree(parent=parent, r=np.asarray(r, dtype=np.float64), res_node=np.asarray(res_node, dtype=np.int32),
                      edge_sign=np.ones(len(parent)))


def star(n, seed=0):
    """One root with n children, one residence on each: a level of n nodes under a single parent."""
    rng = np.random.default_rng(seed)
    parent = np.r_[-1, np.zeros(n, dtype=np.int64)]
    r = np.r_[0.004 / n, 1e-3 * rng.lognormal(0.0, 1.0, n)]
    return _tree(parent, r, np.arange(1, n + 1))


def wide2(m=600, seed=1):
    """Root, m transformers, two residences on each: two wide levels in a row.  Transformer k's children sit at 2k,
    2k + 1 of the last level, so the up pass reads children beyond 512 from parents below it and the down pass reads
    parents beyond 512."""
    rng = np.random.default_rng(seed)
    n = 2 * m
    parent = np.r_[-1, np.zeros(m, dtype=np.int64), 1 + np.repeat(np.arange(m), 2)]
    r = np.r_[0.003 / n, 1e-3 * rng.lognormal(0.0, 0.6, m), 1e-3 * rng.lognormal(0.0, 1.0, n)]
    return _tree(parent, r, np.arange(1 + m, 1 + m + n))


def deep(levels, seed=2, n_zero=7):
    """A trunk chain, a residence on a short lateral at every trunk node: `levels` levels after contraction.  n_zero
    trunk edges of zero resistance (contracted into the node above) and every fifth lateral two edges long, except
    near the end of the trunk, which fixes the depth."""
    rng = np.random.default_rng(seed)
    L = levels - 1                                   # trunk nodes that survive contraction
    zero = set((1 + rng.choice(L - 2, n_zero, replace=False)).tolist())
    parent, r, res = [], [], []
    trunk_r = 0.02 / L ** 2
    prev, depth = -1, -1
    for i in range(L + n_zero):
        parent.append(prev)
        if i in zero:
            r.append(0.0)
        else:
            r.append(trunk_r * rng.lognormal(0.0, 0.3))
            depth += 1
        prev = len(parent) - 1
        at = prev
        if i % 5 == 3 and depth <= L - 3:           # a pole before the service line
            parent.append(at)
            r.append(2e-5 * rng.lognormal(0.0, 0.5))
            at = len(parent) - 1
        parent.append(at)
        r.append(1e-4 * rng.lognormal(0.0, 1.0))
        res.append(len(parent) - 1)
    return _tree(parent, r, res)


def forest(m=700, seed=3):
    """m roots, each a single node with 1..3 residences on it, edge resistances log-uniform over 1e-9..1e-1: R is block
    diagonal with constant blocks (identical rows within a node).  With the targets below only nodes above about 1e-3
    bind (two decades); the other six decades are rows that never bind next to ones that do in one zone.  No node has
    a parent, so a pin cannot form; the warm start at 1e3 times the multipliers holds binding roots whose homes are all
    at zero, which is where "a pin without a parent cannot bind" applies (counted on the host model in
    test_tree_newton_model.py)."""
    rng = np.random.default_rng(seed)
    r = 10.0 ** rng.uniform(-9.0, -1.0, m)
    res = np.repeat(np.arange(m), rng.integers(1, 4, m))
    return _tree(np.full(m, -1), r, res)


def odd_wide(m=560, seed=4):
    """Root, m transformers (level 1), 1..3 residences per transformer (level 2), some daisy-chained behind another
    (level 3), with every irregularity of real feeders at once: residences sharing a node, zero-length service lines
    (the transformer carries a residence and has children), service lines of 1e-22, a zero-length primary edge (its
    residences move up to level 1), a chain of three negligible edges contracted into one transformer, and residences
    behind another one (idle_homes: with z < 0 their rows coincide with the one above and pin it)."""
    rng = np.random.default_rng(seed)
    parent, r, res = [-1], [0.002 / (2.0 * m)], []
    xf = []
    for k in range(m):
        parent.append(0)
        r.append(0.0 if k == 5 else 1e-3 * rng.lognormal(0.0, 0.6))
        xf.append(len(parent) - 1)
        if k == 9:                                   # contracted chain: 1e-22, 0, 1e-22 below the transformer
            for rr in (1e-22, 0.0, 1e-22):
                parent.append(len(parent) - 1)
                r.append(rr)
            xf[-1] = len(parent) - 1
    for k, x in enumerate(xf):
        nh = 1 + k % 3
        for j in range(nh):
            kind = (7 * k + j) % 23
            if kind == 0 and res:                    # shares the node of the previous residence
                res.append(res[-1])
                continue
            parent.append(x)
            r.append(0.0 if kind == 1 else 1e-22 if kind == 2 else 1e-3 * rng.lognormal(0.0, 1.0))
            res.append(len(parent) - 1)
            if kind in (3, 4, 5, 6):                 # a residence behind this one
                parent.append(len(parent) - 1)
                r.append(5e-4 * rng.lognormal(0.0, 0.5))
                res.append(len(parent) - 1)
    return _tree(parent, r, res)


def idle_homes(tr):
    """Residences whose node hangs below another residence's node (daisy chains)."""
    isres = np.zeros(len(tr.parent), bool)
    isres[tr.res_node] = True
    p = tr.parent[tr.res_node]
    return np.nonzero((p >= 0) & isres[np.maximum(p, 0)])[0]


def layout(tr):
    """(levels, widest level, most children of one node, nodes, nodes with several residences) of the zone as
    newton_build_zone lays it out."""
    LT = LevelTree(tr.parent, tr.r, tr.res_node)
    return dict(levels=len(LT.lvl) - 1, widest=int(np.diff(LT.lvl).max()), children=int(LT.nchild.max()), nodes=LT.n,
                shared=int((LT.nhome > 1).sum()))


def _cases():
    return {**{f"star{n}": star(n) for n in (256, 257, 512, 513, 1500)}, "wide2": wide2(),
            **{f"deep{d}": deep(d) for d in (1024, 1025, 2100)}, "forest": forest(), "odd_wide": odd_wide()}


CASES = ["star256", "star257", "star512", "star513", "star1500", "wide2", "deep1024", "deep1025", "deep2100", "forest",
         "odd_wide"]


def _check_layout(name, tr):
    L = layout(tr)
    if name.startswith("star"):
        n = int(name[4:])
        assert L == dict(levels=2, widest=n, children=n, nodes=n + 1, shared=0), L
    elif name == "wide2":
        assert L == dict(levels=3, widest=1200, children=600, nodes=1801, shared=0), L
    elif name.startswith("deep"):
        assert L["levels"] == int(name[4:]) and L["widest"] <= 4 and L["children"] <= 3, L
        assert L["nodes"] < len(tr.parent)          # the zero trunk edges were contracted
    elif name == "forest":
        assert L["levels"] == 1 and L["widest"] == 700 and L["children"] == 0 and L["shared"] > 400, L
    elif name == "odd_wide":
        LT = LevelTree(tr.parent, tr.r, tr.res_node)
        w = np.diff(LT.lvl)
        assert L["levels"] == 4 and w[1] > 512 and w[2] > 512 and L["children"] > 512 and L["shared"] >= 20, L
        assert L["nodes"] < len(tr.parent) - 20     # zero and 1e-22 edges contracted
        assert len(idle_homes(tr)) >= 100
        assert ((LT.nhome > 0) & (LT.nchild > 0)).sum() >= 20      # residences on nodes with children
    return L


@pytest.mark.parametrize("name", CASES)
def test_builder_layout(name):
    """Each builder gives the layout its case exists for (host model of newton_build_zone)."""
    _check_layout(name, _cases()[name])


# ---------------------------------------------------------------------------------------------------------------- data
def targets(tr, T, seed):
    """Targets z [n, T]: base load plus a charger in a share of homes that grows with the column, and idle homes
    (z < 0) behind daisy chains."""
    rng = np.random.default_rng(seed)
    n = tr.n_res
    share = np.linspace(0.15, 0.7, T)
    z = 0.3 + 2.2 * rng.random((n, T)) + 4.8 * (rng.random((n, T)) < share)
    z[idle_homes(tr)] = -0.5
    return z


def forest_projection(tr, z, u):
    """Exact projection for a zone of roots without children: R is rho_k J on the homes of root k, so the problem
    splits into min 1/2 |g - z|^2, g >= 0, sum g <= u / rho per node -- water filling, g = [z - theta]_+.  Returns
    (g, multiplier of each node's row placed on its first home)."""
    rho = 2.0 * tr.r
    g = np.maximum(z, 0.0)
    lam = np.zeros_like(z)
    for k in np.unique(tr.res_node):
        h = np.nonzero(tr.res_node == k)[0]
        cap = u / rho[k]
        for t in range(z.shape[1]):
            zz = z[h, t]
            if np.maximum(zz, 0.0).sum() <= cap:
                continue
            s = np.sort(zz)[::-1]
            cs = np.cumsum(s)
            j = np.arange(1, len(s) + 1)
            th = (cs - cap) / j
            i = np.nonzero(s > th)[0][-1]
            g[h, t] = np.maximum(zz - th[i], 0.0)
            lam[h[0], t] = th[i] / rho[k]
    return g, lam


def _T(name):
    return 4 if name == "deep2100" else 6


def _rres(tr):
    return O.rmat_from_tree(tr.parent, tr.r)[np.ix_(tr.res_node, tr.res_node)]


def _node_homes(tr):
    """(node of every home as the kernel numbers them, the homes that share a node with a lower-numbered home)."""
    LT = LevelTree(tr.parent, tr.r, tr.res_node)
    first = np.zeros(tr.n_res, bool)
    first[np.unique(LT.res, return_index=True)[1]] = True
    return LT.res, ~first


def _spread(lam, node):
    """Each node's multiplier (the sum over its homes) spread evenly over its homes."""
    out = np.empty_like(lam)
    cnt = np.bincount(node)
    for t in range(lam.shape[1]):
        out[:, t] = (np.bincount(node, weights=lam[:, t], minlength=len(cnt)) / np.maximum(cnt, 1))[node]
    return out


def _step(s, z, lam0=None):
    zero = np.zeros_like(z)
    return s.utility_step(2.0 * z, zero, zero, lam0=lam0, **KW)       # target (p_est + p_sch) / 2 = z


# ------------------------------------------------------------------------------------------------------- device checks
@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_projection_on_layout_branches(gpu_lib, name):
    """revs_utility_step on one zone of the shape, every zone on the tree-Newton path: KKT certificate with the device's
    multipliers, the oracle's (or the closed form's) projection per column, multipliers on the first home of a node
    only, warm starts from the device's own multipliers (spread over a node's homes, and 1e3 times too large), and two
    calls give the same bytes."""
    tr = _cases()[name]
    _check_layout(name, tr)
    n, T = tr.n_res, _T(name)
    z = targets(tr, T, seed=11)
    R = _rres(tr)
    node, others = _node_homes(tr)
    with gpu_lib.Solver([n], T) as s:
        s.set_option("newton_min_n", 0)
        s.set_feeder_tree(0, tr.parent, tr.r, tr.res_node)
        g, lam = _step(s, z)
        g2, lam2 = _step(s, z)
        warm = _spread(lam, node)
        gw, lw = _step(s, z, lam0=warm)
        gs, ls = _step(s, z, lam0=1e3 * warm)
    nb = (lam > 0).sum(axis=0)
    assert (nb >= 5).all() and nb.max() >= 60 and nb.max() <= 600, nb          # rows bind, in every column
    kkt_check([R], z, g, lam, U, f"{name} cold")
    assert g.tobytes() == g2.tobytes() and lam.tobytes() == lam2.tobytes(), name
    assert (lam[others] == 0.0).all(), (name, "multiplier off the first home of its node")
    for tag, (gg, ll) in (("warm", (gw, lw)), ("warm x1e3", (gs, ls))):
        kkt_check([R], z, gg, ll, U, f"{name} {tag}")
        assert (ll[others] == 0.0).all(), (name, tag)
        assert np.abs(gg - g).max() <= 1e-8, (name, tag, np.abs(gg - g).max())
    if name == "forest":
        gf, lf = forest_projection(tr, z, U)
        assert np.abs(g - gf).max() <= 1e-8, np.abs(g - gf).max()
        act = lf > 0
        assert np.abs(lam[act] - lf[act]).max() <= 1e-6 * np.abs(lf[act]).max()
        assert not (lam[~act] > 0).any()
    else:
        for t in range(T):
            g0, _, _ = O.project_voltage(z[:, t], R, U)
            assert np.abs(g[:, t] - g0).max() <= 1e-8, (name, t, np.abs(g[:, t] - g0).max())
    if name == "odd_wide":       # idle residences behind binding ones: duplicate binding rows the kernel turns into pins
        idle = idle_homes(tr)
        v = R @ g
        assert (np.abs(v[idle] - U) <= 1e-9).sum(axis=0).min() >= 5


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_zone_alone_and_among_others(gpu_lib, name):
    """The zone alone, and the same zone after two small tree-Newton zones and one dense zone in one solver, give the
    same bytes of g and lam: a column reads only its own zone, whatever the other zones' layout and targets."""
    from revs_admm_b200.feeder import synthetic_feeder
    tr = _cases()[name]
    n, T = tr.n_res, _T(name)
    z = targets(tr, T, seed=12)
    with gpu_lib.Solver([n], T) as s:
        s.set_option("newton_min_n", 0)
        s.set_feeder_tree(0, tr.parent, tr.r, tr.res_node)
        g, lam = _step(s, z)
    others = [synthetic_feeder(k, seed=k, r_secondary=1e-3, laterals=3) for k in (40, 300, 90)]
    sizes = [t.n_res for t in others] + [n]
    rng = np.random.default_rng(5)
    zo = 6.0 * rng.random((sum(sizes[:3]), T))
    with gpu_lib.Solver(sizes, T) as s:
        s.set_option("newton_min_n", 0)
        s.set_feeder_trees(others + [tr])
        s.set_sensitivity(2, _rres(others[2]))           # zone 2 back on the dense kernels
        ga, la = _step(s, np.vstack([zo, z]))
    sl = slice(sum(sizes[:3]), None)
    assert ga[sl].tobytes() == g.tobytes() and la[sl].tobytes() == lam.tobytes(), name
    assert (la[:sum(sizes[:3])] > 0).any()               # the other zones bind too

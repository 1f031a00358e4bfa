"""CPU checks of the tree-Newton linear algebra (tests/tree_newton_ref.py = host model of csrc/tree_newton.cu) against
dense matrices and against the oracle's projection (oracle.project_voltage, dense R as in lpsolver.py:17-26, 183-194)."""
import numpy as np
import pytest

import revs_oracle as O
import test_gpu_newton_shapes as S
from tree_newton_ref import LevelTree, tree_product, tree_solve

U = 1.05 ** 2 - 1.03 ** 2


def _cases():
    from revs_admm_b200.feeder import radial_feeder, synthetic_feeder, reference_shaped_feeder
    odd = synthetic_feeder(300, seed=5, r_secondary=1e-3)
    odd.res_node[10] = odd.res_node[11]                       # two residences on one node
    odd.res_node[50] = odd.res_node[51] = odd.res_node[52]
    odd.r[odd.res_node[100]] = 0.0                            # zero-length service line
    odd.r[3] = 0.0                                            # zero-length primary edge
    odd.r[odd.res_node[200]] = 1e-22
    return {"radial": radial_feeder(700, seed=2), "laterals": synthetic_feeder(600, seed=0, laterals=3),
            "refshape": reference_shaped_feeder(500, seed=4), "odd": odd,
            # shapes of the device kernel's layout branches (tests/test_gpu_newton_shapes.py)
            "star513": S.star(513), "wide2": S.wide2(), "deep1025": S.deep(1025), "forest": S.forest(),
            "odd_wide": S.odd_wide()}


def test_product_and_elimination_match_dense_matrices():
    from revs_admm_b200.feeder import radial_feeder
    tr = radial_feeder(400, seed=1)
    N = len(tr.parent)
    rho = 2.0 * tr.r
    Rf = O.rmat_from_tree(tr.parent, tr.r)
    rng = np.random.default_rng(0)
    x = rng.random(N)
    assert np.abs(tree_product(tr.parent, rho, x) - Rf @ x).max() <= 1e-15 * np.abs(Rf @ x).max()
    isres = np.zeros(N, bool)
    isres[tr.res_node] = True
    z = np.zeros(N)
    z[tr.res_node] = rng.lognormal(0.5, 0.6, tr.n_res)
    F = isres & (rng.random(N) < 0.8)
    A = F & (rng.random(N) < 0.3)
    s = 1e-14
    xx, mu, g, v = tree_solve(tr.parent, rho, z, F, A, np.full(N, U), s)
    RAF = Rf[np.ix_(A, F)]
    xd = np.linalg.solve(RAF @ RAF.T + s * np.eye(A.sum()), RAF @ z[F] - U)
    assert np.abs(xx[A] - xd).max() <= 1e-9 * np.abs(xd).max()
    assert np.abs(v - Rf @ g).max() <= 1e-12
    LT = LevelTree(tr.parent, tr.r, tr.res_node, contract=False)
    xo = np.zeros(N)
    xo[LT.order] = x
    assert np.abs(LT.product(x) - (Rf @ xo)[LT.order]).max() <= 1e-15 * np.abs(Rf @ x).max()


@pytest.mark.parametrize("name", ["radial", "laterals", "refshape", "odd", "star513", "wide2", "deep1025", "forest", "odd_wide"])
def test_tree_projection_equals_oracle_projection(name):
    from revs_admm_b200.feeder import synthetic_homes
    tr = _cases()[name]
    n = tr.n_res
    LT = LevelTree(tr.parent, tr.r, tr.res_node)
    R = O.rmat_from_tree(tr.parent, tr.r)[np.ix_(tr.res_node, tr.res_node)]
    hm = synthetic_homes(n, 96, seed=3)
    rng = np.random.default_rng(0)
    lam_prev = None
    for tcol in (0, 52):
        z = hm["load"][:, tcol] + hm["has_ev"] * 4.8 * (rng.random(n) < 0.6)
        g0, l0, _ = O.project_voltage(z, R, U)
        st = {}
        g1, l1, _ = LT.project(z, U, lam0_res=lam_prev, stats=st)
        lam_prev = l1
        assert np.abs(g0 - g1).max() <= 1e-9
        assert (R @ g1 - U).max() <= 1e-10                                     # KKT certificate, independent of either solver
        assert np.abs(g1 - np.maximum(z - R @ l1, 0.0)).max() <= 1e-9
        assert np.abs(l1 * (U - R @ g1)).max() <= 1e-8
        assert st["solves"] <= (400 if name == "deep1025" else 60)        # a 1024-node chain: guesses reshuffle rows along it


def test_forest_closed_form_equals_oracle_projection():
    """The water-filling projection of a zone of roots without children (the reference of the device's forest case)
    is the oracle's projection, on nodes that bind (edge resistances from about 2e-3 to 1e-1: with these targets no
    node below about 1e-3 can reach the limit) and on nodes that do not."""
    tr = S.forest()
    z = S.targets(tr, 3, seed=11)
    z[::17] = -0.3                                        # homes at zero next to binding ones on the same node
    g, lam = S.forest_projection(tr, z, U)
    R = O.rmat_from_tree(tr.parent, tr.r)[np.ix_(tr.res_node, tr.res_node)]
    for t in range(z.shape[1]):
        g0, l0, _ = O.project_voltage(z[:, t], R, U)
        assert np.abs(g[:, t] - g0).max() <= 1e-9
        node = np.bincount(tr.res_node, weights=l0, minlength=len(tr.parent))
        act = node > 0
        assert 50 <= act.sum() <= 300
        assert tr.r[act].min() <= 3e-3 and tr.r[act].max() >= 5e-2          # binding nodes over almost two decades
        assert np.abs(np.bincount(tr.res_node, weights=lam[:, t], minlength=len(tr.parent)) - node).max() <= 1e-6 * node.max()
    assert (R @ g - U).max() <= 1e-10


def test_forest_warm_start_reaches_the_parentless_pin_rule(monkeypatch):
    """A row whose subtree holds no home of the piece pins its parent; a root has none, so its row sits the guess out
    ("a pin without a parent cannot bind").  The device's forest case reaches that rule through its warm start at 1e3
    times the multipliers: the first guesses hold binding roots whose homes are all at zero.  Counted here on the host
    model, which runs the same iteration; the projection still equals the closed form."""
    import tree_newton_ref as TR
    tr = S.forest()
    z = S.targets(tr, 2, seed=11)
    gf, lf = S.forest_projection(tr, z, U)
    LT = LevelTree(tr.parent, tr.r, tr.res_node)
    hits = []
    solve = TR.LevelTree.solve

    def counting(self, nF, zF, A, t, s):
        hits.append(int((A & (nF == 0) & (self.nchild == 0) & (self.parent < 0)).sum()))
        return solve(self, nF, zF, A, t, s)

    monkeypatch.setattr(TR.LevelTree, "solve", counting)
    for col in range(z.shape[1]):
        hits.clear()
        g, _, _ = LT.project(z[:, col], U, lam0_res=lf[:, col])
        assert sum(hits) == 0 and np.abs(g - gf[:, col]).max() <= 1e-9
        g, _, _ = LT.project(z[:, col], U, lam0_res=1e3 * lf[:, col])
        assert sum(hits) >= 50 and np.abs(g - gf[:, col]).max() <= 1e-9


def test_tree_projection_on_the_reference_feeder_as_one_zone(case121144):
    """Network 121144 unsplit (1126 residences, primary edges of 1e-20, idle homes below binding rows)."""
    from revs_admm_b200 import lpsolver
    from revs_admm_b200.feeder import tree_from_graph
    c = case121144
    tree = tree_from_graph(c["dist"])
    arr = lpsolver._home_arrays(c["homes"], list(tree.res_ids))
    LT = LevelTree(tree.parent, tree.r, tree.res_node)
    assert LT.n < len(tree.parent)                 # the negligible edges were contracted
    R = O.rmat_from_tree(tree.parent, tree.r)[np.ix_(tree.res_node, tree.res_node)]
    rng = np.random.default_rng(0)
    for tcol in (9, 12):
        z = arr["load"][:, tcol] + arr["has_ev"] * 4.8 * (rng.random(tree.n_res) < 0.5)
        g0, _, _ = O.project_voltage(z, R, U)
        g1, l1, _ = LT.project(z, U)
        assert np.abs(g0 - g1).max() <= 1e-9
        assert np.abs(g1 - np.maximum(z - R @ l1, 0.0)).max() <= 1e-9

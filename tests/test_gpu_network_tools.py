"""GPU: the network check, the repair, the bracket and the certificate share one set of device scratch.  Each call gives
the bytes it gives on a fresh solver whatever ran before it on the same solver, the kept schedules (network_check of
"repaired" and "central") survive the other tools' calls, and the ADMM run's results and estimate stay as they are."""
import numpy as np
import pytest

import network_ref as NR
from revs_admm_b200.feeder import FeederTree, population, radial_feeder, synthetic_homes, synthetic_tariff
from test_gpu_network import _mixed_zones, _solver

pytestmark = pytest.mark.gpu

T = 96
ADMM = dict(kappa=5.0, iter_max=4, vset=1.0, vlow=0.95, vhigh=1.05)
KEPT = {"repair": "repaired", "bracket": "central"}      # the tool whose call makes a network_check source valid


def _population():
    """Mixed zones, reference-shaped zones and a 2,300-residence tree-only zone, whose repair state lives in the global
    scratch.  Every zone's resistances are scaled so that its base load alone reaches a given share of the limit (over
    it for some zones), so that every tool has work in zones of every shape."""
    ref, ref_hm, _, _, t_ref = population("refshape", 2, seed=0)
    assert t_ref == T
    zones = _mixed_zones(T) + ref + [radial_feeder(2300, seed=3, r_scale=0.07)]
    parts = [synthetic_homes(sum(z.n_res for z in zones[:4]), T, seed=T), ref_hm, synthetic_homes(2300, T, seed=4)]
    hm = {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
    u = 0.01
    drop = NR.network_check(zones, hm["load"])["zone_worst"][:, 0]
    share = np.resize([0.6, 0.75, 0.9, 1.1], len(zones))
    share[-1] = 0.5                  # over the limit after the ADMM run, but a short repair
    zones = [FeederTree(parent=z.parent, r=z.r * (f * u / d), res_node=z.res_node) for z, f, d in zip(zones, share, drop)]
    return zones, hm, synthetic_tariff(T), dict(vset=1.0, vhigh=float(np.sqrt(1.0 + u)))


def _assert_same(a, b, what):
    assert a.keys() == b.keys(), what
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes(), (what, k)
        else:
            assert a[k] == b[k], (what, k)


def test_calls_keep_their_bytes_in_any_order(gpu_lib):
    zones, hm, cost, lim = _population()
    P = np.random.default_rng(7).uniform(0.0, 2.0, (len(hm["load"]), T))
    calls = {"host": lambda s: s.network_check(P, vlow=0.9, full=True, zones=True, **lim),
             "repair": lambda s: s.repair_schedule(mask=True, **lim),
             "bracket": lambda s: s.central_bracket(mask=True, iters=10, **lim),
             "certify": lambda s: s.certify_infeasible(**lim)}

    def ready():
        s = _solver(gpu_lib, zones, T)
        s.set_homes(**hm)
        s.set_tariff(cost)
        return s

    ref, kept = {}, {}
    for name, call in calls.items():
        with ready() as s:
            if name == "repair":
                s.solve_admm(**ADMM)
            ref[name] = call(s)
            if name in KEPT:
                kept[KEPT[name]] = s.network_check(KEPT[name], zones=True, **lim)
    assert ref["repair"]["zone_info"][-1, 0] > 0 and ref["bracket"]["zone_info"][-1, 0] > 0    # the tree-only zone
    assert ref["certify"]["certified"] > 0

    first = ["certify", "bracket", "admm", "repair", "host", "bracket", "repair", "certify"]
    second = ["host", "repair", "certify", "bracket", "host"]
    with ready() as s:
        valid, admm = set(), None
        for step, name in enumerate(first + second):
            if name == "admm":
                s.solve_admm(**ADMM)
                valid.discard("repaired")
                admm = s.results(), s.estimate()
            else:
                _assert_same(calls[name](s), ref[name], (step, name))
                valid |= {KEPT[name]} if name in KEPT else set()
            for src in sorted(valid):
                _assert_same(s.network_check(src, zones=True, **lim), kept[src], (step, name, src))
            if admm is not None:
                res, est = s.results(), s.estimate()
                _assert_same(res, admm[0], (step, name, "results"))
                assert all(a.tobytes() == b.tobytes() for a, b in zip(est, admm[1])), (step, name, "estimate")

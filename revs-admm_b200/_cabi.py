"""ctypes binding of include/revs_admm.h.  No torch types cross this boundary.

The library is the product: if it is missing or no B200 is visible every call raises --
there is no CPU path in this package.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("REVS_LIB") or os.path.join(HERE, "librevs_admm.so")     # REVS_LIB: a build variant (profiles/build_variants.sh)

REVS_REL_VOLTAGE, REVS_REL_FLOW, REVS_REL_DROP = 0, 1, 2
REVS_NET_SCHEDULE, REVS_NET_ESTIMATE, REVS_NET_HOST, REVS_NET_REPAIRED, REVS_NET_CENTRAL = 0, 1, 2, 3, 4


class RevsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"revs_admm error {code}: {msg}")
        self.code = code


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("gemm_launches", C.c_int64), ("gemm_full_launches", C.c_int64),
                ("qp_outer_iterations", C.c_int64), ("qp_newton_iterations", C.c_int64),
                ("admm_iterations", C.c_int32), ("max_working_set", C.c_int32),
                ("primal_residual", C.c_double), ("dual_residual", C.c_double), ("qp_flops", C.c_double),
                ("gemm_ms", C.c_float), ("gemm_full_ms", C.c_float), ("home_ms", C.c_float), ("dual_ms", C.c_float),
                ("qp_ms", C.c_float), ("qp_big_ms", C.c_float), ("total_ms", C.c_float),
                ("qp_warp_ms", C.c_float), ("qp_init_ms", C.c_float), ("qp_columns", C.c_int64),
                ("qp_warp_rounds", C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class NetworkSummary(C.Structure):
    """revs_network_summary: worst voltage drop, voltage-row excess and line loading of a population, where they
    are (zone, node or residence local to its zone, step) and the violation counts."""
    _fields_ = [("drop_max", C.c_double), ("v_min", C.c_double),
                ("drop_zone", C.c_int32), ("drop_node", C.c_int32), ("drop_step", C.c_int32), ("pad0_", C.c_int32),
                ("row_excess_max", C.c_double),
                ("excess_zone", C.c_int32), ("excess_res", C.c_int32), ("excess_step", C.c_int32), ("pad1_", C.c_int32),
                ("rows_violated", C.c_int64), ("nodes_below_vlow", C.c_int64), ("loading_max", C.c_double),
                ("loading_zone", C.c_int32), ("loading_node", C.c_int32), ("loading_step", C.c_int32), ("pad2_", C.c_int32),
                ("edges_overloaded", C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if not k.startswith("pad")}


_P = C.c_void_p
_D = C.POINTER(C.c_double)
# name -> argtypes   (every symbol include/revs_admm.h declares)
SIGNATURES = {
    "revs_last_error": ([], C.c_char_p),
    "revs_version": ([], C.c_int),
    "revs_device_count": ([C.POINTER(C.c_int)], C.c_int),
    "revs_create": ([C.POINTER(_P), C.c_int, C.c_int, C.POINTER(C.c_int64), C.c_int], C.c_int),
    "revs_destroy": ([_P], C.c_int),
    "revs_set_sensitivity": ([_P, C.c_int, _D], C.c_int),
    "revs_set_feeder_tree": ([_P, C.c_int, C.c_int, C.POINTER(C.c_int32), _D, C.POINTER(C.c_int32)], C.c_int),
    "revs_set_feeder_trees": ([_P, C.POINTER(C.c_int64), C.POINTER(C.c_int32), _D, C.POINTER(C.c_int32)], C.c_int),
    "revs_set_homes": ([_P, _D, C.POINTER(C.c_uint8), _D, _D, _D, C.POINTER(C.c_int32),
                        C.POINTER(C.c_int32)], C.c_int),
    "revs_set_tariff": ([_P, _D], C.c_int),
    "revs_solve_admm": ([_P, C.c_double, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double,
                         C.POINTER(C.c_int)], C.c_int),
    "revs_admm_begin": ([_P, C.c_double, C.c_int, C.c_double, C.c_double, C.c_double], C.c_int),
    "revs_admm_step": ([_P, _D], C.c_int),
    "revs_home_step": ([_P, C.c_double, _D, _D, _D, _D, _D], C.c_int),
    "revs_utility_step": ([_P, C.c_double, C.c_double, C.c_double, C.c_double, _D, _D, _D, _D, _D, _D], C.c_int),
    "revs_get_results": ([_P, _D, _D, _D, _D, C.c_int], C.c_int),
    "revs_get_schedule": ([_P, _D, C.POINTER(C.c_uint64), C.c_int, _D, C.c_int], C.c_int),
    "revs_get_schedule_ld": ([_P, _D, C.POINTER(C.c_uint64), C.c_int, _D, C.c_int, C.c_int64], C.c_int),
    "revs_get_estimate": ([_P, _D, _D], C.c_int),
    "revs_solve_individual": ([_P, _D, _D, _D], C.c_int),
    "revs_reliability": ([_P, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), _D, C.c_double, _D, _D], C.c_int),
    "revs_contract": ([C.c_int, C.c_int, C.c_int, C.c_int, _D, _D, _D], C.c_int),
    "revs_set_option": ([_P, C.c_char_p, C.c_double], C.c_int),
    "revs_screen_contract": ([C.c_int, C.c_int, C.c_int, C.c_int, _D, _D, _D, C.c_int], C.c_int),
    "revs_get_stats": ([_P, C.POINTER(Stats)], C.c_int),
    "revs_comm_export": ([_P, C.c_void_p], C.c_int),
    "revs_comm_attach": ([_P, C.c_int, C.c_int, C.c_void_p], C.c_int),
    "revs_comm_detach": ([_P], C.c_int),
    "revs_gather_export": ([_P, C.c_int64, C.c_void_p], C.c_int),
    "revs_gather_attach": ([_P, C.c_int, C.c_int, C.c_void_p], C.c_int),
    "revs_reliability_sharded": ([_P, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), _D, C.c_double, _D, _D], C.c_int),
    "revs_network_check": ([_P, C.c_int, _D, C.c_double, C.c_double, C.c_double, C.c_double, _D, _D, _D, _D,
                            C.POINTER(NetworkSummary)], C.c_int),
    "revs_repair_schedule": ([_P, C.c_double, C.c_double, C.c_double, _D, C.POINTER(C.c_uint64), C.c_int,
                              C.POINTER(C.c_int32)], C.c_int),
    "revs_central_bracket": ([_P, C.c_double, C.c_double, C.c_double, C.c_int, _D, C.POINTER(C.c_uint64), C.c_int, _D,
                              C.POINTER(C.c_int32)], C.c_int),
    "revs_certify_infeasible": ([_P, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_int32), C.POINTER(C.c_int)],
                                C.c_int),
    "revs_hosting_capacity": ([_P, C.c_int, _D, C.c_double, C.c_double, C.c_double, _D, _D, _D, C.POINTER(C.c_int64)],
                              C.c_int),
}

_lib = None


def load():
    """dlopen the in-tree library and type every entry point."""
    global _lib
    if _lib is None:
        path = os.environ.get("REVS_LIB") or LIB_PATH        # REVS_LIB: another build of this library (A/B measurements)
        if not os.path.exists(path):
            raise RevsError(-1, f"{path} is missing -- run `python revs-admm_b200/_build.py` "
                                "(there is no CPU fallback)")
        lib = C.CDLL(path)
        for name, (args, res) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes, fn.restype = args, res
        _lib = lib
    return _lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(_D)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and a.shape != tuple(shape):
        raise ValueError(f"expected shape {tuple(shape)}, got {a.shape}")
    return a


def _check(rc):
    if rc != 0:
        raise RevsError(rc, load().revs_last_error().decode())


def device_count():
    n = C.c_int(0)
    _check(load().revs_device_count(C.byref(n)))
    return n.value


def contract(A, B, device=0):
    """C = A @ B through the FP64 tensor-core contraction kernel (host in/out)."""
    A, B = _f64(A), _f64(B)
    M, K = A.shape
    K2, T = B.shape
    assert K == K2
    out = np.empty((M, T))
    _check(load().revs_contract(device, M, K, T, _dp(A), _dp(B), _dp(out)))
    return out


def screen_contract(A, B, impl=0, device=0):
    """C ~ A @ B through the BF16 screening kernel (impl 0: mma.sync, 1: tcgen05/TMA)."""
    A, B = _f64(A), _f64(B)
    M, K = A.shape
    K2, T = B.shape
    assert K == K2
    out = np.empty((M, T))
    _check(load().revs_screen_contract(device, M, K, T, _dp(A), _dp(B), _dp(out), impl))
    return out


def expand_schedule(mask, T, has_ev, rating, capacity, initial):
    """P_ev [H,T] and SOC [H,T+1] (the S and C of lpsolver.py:289-290) from the charging bit masks of
    Solver.schedule_compact and the per-home inputs: P_ev = rating * bit, SOC[t+1] = SOC[t] + P_ev[t] / capacity
    (same operation order as the device kernel, so bit-identical with Solver.results)."""
    mask = np.asarray(mask, dtype=np.uint64)
    H = mask.shape[0]
    t = np.arange(T)
    bits = ((mask[:, t // 64] >> (t % 64).astype(np.uint64)) & np.uint64(1)).astype(bool)
    ev = np.asarray(has_ev).astype(bool)
    p_ev = np.where(bits & ev[:, None], np.asarray(rating, dtype=np.float64)[:, None], 0.0)
    soc = np.zeros((H, T + 1))
    soc[:, 0] = np.where(ev, initial, 0.0)
    inc = p_ev / np.where(ev, capacity, 1.0)[:, None]
    for k in range(T):
        soc[:, k + 1] = soc[:, k] + inc[:, k]
    return p_ev, soc


def repair_totals(r):
    """Add the totals of zone_info to a repair_schedule result."""
    z = r["zone_info"]
    r.update(moves=int(z[:, 1].sum()), drops=int(z[:, 2].sum()), zones_violated=int((z[:, 0] > 0).sum()),
             zones_repaired=int((z[:, 0] == 1).sum()), zones_left=int((z[:, 0] == 2).sum()))
    return r


def central_totals(r):
    """Add the totals of zone_bounds / zone_info to a central_bracket result: lb (sum of LB over all zones), lb_bracketed
    and ub (sums of LB and UB over the zones of status 0 and 1), gap = (ub - lb_bracketed) / |lb_bracketed| and
    zones_status (zones of status 0, 1, 2, 3)."""
    b, st = r["zone_bounds"], r["zone_info"][:, 0]
    ok = st <= 1
    lbb, ub = float(b[ok, 0].sum()), float(b[ok, 1].sum())
    r.update(lb=float(b[:, 0].sum()), lb_bracketed=lbb, ub=ub, gap=(ub - lbb) / abs(lbb) if lbb else 0.0,
             zones_status=[int((st == k).sum()) for k in range(4)])
    return r


def certify_totals(r):
    """Add the counts of zone_cert to a certify_infeasible result: zones_kind (zones of kind 0, 1, 2) and certified
    (zones of kind 1 or 2)."""
    kind = r["zone_cert"][:, 0]
    r.update(zones_kind=[int((kind == k).sum()) for k in range(3)], certified=int((kind > 0).sum()))
    return r


def hosting_totals(r, zone_off):
    """Add the totals of a hosting_capacity result: window_steps, window_steps_open and thermal_bound (zone_counts summed
    over the zones), home_cap_min = dict(value, zone, index, step) of the smallest home capacity (index local to the
    zone; zone_off = the [zones + 1] home offsets) and uniform_min = dict(value, zone, step) of the smallest uniform
    headroom.  Ties go to the lowest zone, index, step; a minimum is None when its array was not asked for."""
    c = r["zone_counts"]
    r.update(window_steps=int(c[:, 0].sum()), window_steps_open=int(c[:, 1].sum()), thermal_bound=int(c[:, 2].sum()),
             home_cap_min=None, uniform_min=None)
    cap, uni = r["home_cap"], r["zone_uniform"]
    if cap is not None and cap.size:
        k = int(np.argmin(cap))
        h, t = divmod(k, cap.shape[1])
        z = int(np.searchsorted(zone_off, h, side="right")) - 1
        r["home_cap_min"] = dict(value=float(cap.flat[k]), zone=z, index=h - int(zone_off[z]), step=t)
    if uni is not None and uni.size:
        k = int(np.argmin(uni))
        z, t = divmod(k, uni.shape[1])
        r["uniform_min"] = dict(value=float(uni.flat[k]), zone=z, step=t)
    return r


def central_status(zone_info, zone_cert):
    """The status of central_bracket's zone_info with the zones that certify_infeasible proves infeasible: 2 (no feasible
    schedule found) becomes 3 (certified infeasible) where zone_cert has a certificate.  Raises ValueError when a zone
    of status 0 or 1 (a voltage-feasible schedule is known) is certified: one of the two results would be wrong."""
    st = np.array(np.asarray(zone_info)[:, 0], dtype=np.int32)
    cert = np.asarray(zone_cert)[:, 0] > 0
    bad = np.nonzero(cert & (st <= 1))[0]
    if bad.size:
        raise ValueError(f"zones {bad.tolist()} have a voltage-feasible schedule and a certificate of infeasibility")
    st[cert] = 3
    return st


class Solver:
    """A batch of feeders resident on one GPU (wraps revs_solver*)."""

    def __init__(self, feeder_sizes, T, device=0):
        self.lib = load()
        self.sizes = [int(n) for n in feeder_sizes]
        self.off = np.concatenate([[0], np.cumsum(self.sizes)]).astype(np.int64)
        self.H, self.T, self.nf = int(self.off[-1]), int(T), len(self.sizes)
        self.node_counts = [None] * self.nf        # nodes of every zone's tree, as given to set_feeder_tree(s)
        self._h = _P()
        _check(self.lib.revs_create(C.byref(self._h), device, self.nf,
                                    self.off.ctypes.data_as(C.POINTER(C.c_int64)), self.T))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.revs_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- inputs
    def set_sensitivity(self, feeder, R):
        n = self.sizes[feeder]
        R = _f64(R, (n, n))
        _check(self.lib.revs_set_sensitivity(self._h, feeder, _dp(R)))

    def set_feeder_tree(self, feeder, parent, r, res_node):
        parent = np.ascontiguousarray(parent, dtype=np.int32)
        r = _f64(r, (len(parent),))
        res_node = np.ascontiguousarray(res_node, dtype=np.int32)
        assert len(res_node) == self.sizes[feeder]
        i32 = C.POINTER(C.c_int32)
        _check(self.lib.revs_set_feeder_tree(self._h, feeder, len(parent), parent.ctypes.data_as(i32),
                                             _dp(r), res_node.ctypes.data_as(i32)))
        self.node_counts[feeder] = len(parent)

    def pack_trees(self, trees):
        """The concatenated arrays revs_set_feeder_trees takes, from feeder.FeederTree-like objects (parent, r, res_node)."""
        assert len(trees) == self.nf
        node_off = np.concatenate([[0], np.cumsum([len(t.parent) for t in trees])]).astype(np.int64)
        parent = np.ascontiguousarray(np.concatenate([t.parent for t in trees]), dtype=np.int32)
        r = _f64(np.concatenate([t.r for t in trees]))
        res = np.ascontiguousarray(np.concatenate([t.res_node for t in trees]), dtype=np.int32)
        assert len(res) == self.H
        return node_off, parent, r, res

    def set_feeder_trees(self, trees, packed=None):
        """All feeders in one call; `trees` are feeder.FeederTree-like (parent, r, res_node), or `packed` = pack_trees(trees)."""
        node_off, parent, r, res = packed if packed is not None else self.pack_trees(trees)
        i32 = C.POINTER(C.c_int32)
        _check(self.lib.revs_set_feeder_trees(self._h, node_off.ctypes.data_as(C.POINTER(C.c_int64)),
                                              parent.ctypes.data_as(i32), _dp(r), res.ctypes.data_as(i32)))
        self.node_counts = np.diff(node_off).astype(int).tolist()

    def set_homes(self, load, has_ev, rating, capacity, initial, start, end):
        H, T = self.H, self.T
        load = _f64(load, (H, T))
        has_ev = np.ascontiguousarray(has_ev, dtype=np.uint8)
        rating, capacity, initial = _f64(rating, (H,)), _f64(capacity, (H,)), _f64(initial, (H,))
        start = np.ascontiguousarray(start, dtype=np.int32)
        end = np.ascontiguousarray(end, dtype=np.int32)
        i32 = C.POINTER(C.c_int32)
        _check(self.lib.revs_set_homes(self._h, _dp(load), has_ev.ctypes.data_as(C.POINTER(C.c_uint8)),
                                       _dp(rating), _dp(capacity), _dp(initial),
                                       start.ctypes.data_as(i32), end.ctypes.data_as(i32)))

    def set_tariff(self, cost):
        cost = _f64(cost, (self.T,))
        _check(self.lib.revs_set_tariff(self._h, _dp(cost)))

    # ---- solves
    def solve_admm(self, kappa=5.0, iter_max=15, vset=1.0, vlow=0.95, vhigh=1.05, tol=0.0):
        done = C.c_int(0)
        _check(self.lib.revs_solve_admm(self._h, kappa, iter_max, vset, vlow, vhigh, tol, C.byref(done)))
        return done.value

    def admm_begin(self, kappa=5.0, iter_max=15, vset=1.0, vlow=0.95, vhigh=1.05):
        _check(self.lib.revs_admm_begin(self._h, kappa, iter_max, vset, vlow, vhigh))

    def admm_step(self):
        sums = np.zeros(3)
        _check(self.lib.revs_admm_step(self._h, _dp(sums)))
        return sums

    def home_step(self, p_est, p_sch, gamma, kappa=5.0):
        H, T = self.H, self.T
        g, p = np.empty((H, T)), np.empty((H, T))
        _check(self.lib.revs_home_step(self._h, kappa, _dp(_f64(p_est, (H, T))), _dp(_f64(p_sch, (H, T))),
                                       _dp(_f64(gamma, (H, T))), _dp(g), _dp(p)))
        return g, p

    def utility_step(self, p_est, p_sch, gamma, kappa=5.0, vset=1.0, vlow=0.95, vhigh=1.05, lam0=None):
        H, T = self.H, self.T
        g, lam = np.empty((H, T)), np.empty((H, T))
        l0 = None if lam0 is None else _f64(lam0, (H, T))
        _check(self.lib.revs_utility_step(self._h, kappa, vset, vlow, vhigh, _dp(_f64(p_est, (H, T))),
                                          _dp(_f64(p_sch, (H, T))), _dp(_f64(gamma, (H, T))), _dp(l0),
                                          _dp(g), _dp(lam)))
        return g, lam

    def results(self, iters=None, want_diff=True, out=None):
        """`out`: optional dict of preallocated (e.g. page-locked) arrays P_sch, P_ev, SOC, diff."""
        H, T = self.H, self.T
        done = self.stats()["admm_iterations"]
        iters = done if iters is None else iters
        if out is not None:
            P, E, S, D = out["P_sch"], out["P_ev"], out["SOC"], out.get("diff")
            for a, shape in ((P, (H, T)), (E, (H, T)), (S, (H, T + 1))):
                if a.shape != shape or a.dtype != np.float64 or not a.flags.c_contiguous:
                    raise ValueError(f"out arrays must be C-contiguous float64 of shape {shape}")
            if D is not None and (D.ndim != 2 or D.shape[1] != H or D.dtype != np.float64 or not D.flags.c_contiguous):
                raise ValueError("out['diff'] must be a C-contiguous float64 [rows, H] array")
        else:
            P, E, S = np.empty((H, T)), np.empty((H, T)), np.empty((H, T + 1))
            D = np.empty((max(iters, done), H)) if want_diff else None
        # the library refuses a diff buffer with fewer rows than iterations that ran
        _check(self.lib.revs_get_results(self._h, _dp(P), _dp(E), _dp(S), _dp(D), 0 if D is None else D.shape[0]))
        return dict(P_sch=P, P_ev=E, SOC=S, diff=None if D is None else D[:done] if out is None else D)

    def schedule_compact(self, want_diff=True, out=None):
        """P_sch, the charging decisions as bit masks [H, ceil(T/64)] (uint64) and diff -- a third of the
        bytes of results(); expand_schedule() rebuilds P_ev and SOC from the mask on the host."""
        H, T = self.H, self.T
        W = (T + 63) // 64
        done = self.stats()["admm_iterations"]
        if out is None:
            out = dict(P_sch=np.empty((H, T)), mask=np.empty((H, W), dtype=np.uint64),
                       diff=np.empty((done, H)) if want_diff else None)
        P, M, D = out["P_sch"], out["mask"], out.get("diff")
        if P.shape != (H, T) or P.dtype != np.float64 or not P.flags.c_contiguous:
            raise ValueError("out['P_sch'] must be a C-contiguous float64 [H, T] array")
        if M.shape != (H, W) or M.dtype != np.uint64 or not M.flags.c_contiguous:
            raise ValueError("out['mask'] must be a C-contiguous uint64 [H, ceil(T/64)] array")
        # diff may be a column block of a wider [rows, all homes] array (rows strided, elements contiguous): the
        # library writes it in place (revs_get_schedule_ld)
        ld = H
        if D is not None:
            if D.ndim != 2 or D.shape[1] != H or D.dtype != np.float64 or (H > 1 and D.strides[1] != 8) or \
                    (D.shape[0] > 1 and (D.strides[0] % 8 or D.strides[0] < 8 * H)):
                raise ValueError("out['diff'] must be a float64 [rows, H] array with contiguous rows")
            ld = D.strides[0] // 8 if D.shape[0] > 1 else H
        dptr = _dp(D)
        _check(self.lib.revs_get_schedule_ld(self._h, _dp(P), M.ctypes.data_as(C.POINTER(C.c_uint64)), W, dptr,
                                             0 if D is None else D.shape[0], ld))
        return dict(P_sch=P, mask=M, diff=D)

    def estimate(self):
        H, T = self.H, self.T
        P, G = np.empty((H, T)), np.empty((H, T))
        _check(self.lib.revs_get_estimate(self._h, _dp(P), _dp(G)))
        return P, G

    def solve_individual(self):
        H, T = self.H, self.T
        P, E, S = np.empty((H, T)), np.empty((H, T)), np.empty((H, T + 1))
        _check(self.lib.revs_solve_individual(self._h, _dp(P), _dp(E), _dp(S)))
        return dict(P_res=P, P_ev=E, SOC=S)

    def reliability(self, feeder, kind, rows, vset=1.0, scale=None, P=None):
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        out = np.empty((len(rows), self.T))
        sc = None if scale is None else _f64(scale, (len(rows),))
        Pp = None if P is None else _f64(P, (self.sizes[feeder], self.T))
        _check(self.lib.revs_reliability(self._h, feeder, kind, len(rows),
                                         rows.ctypes.data_as(C.POINTER(C.c_int32)), _dp(sc), vset,
                                         _dp(Pp), _dp(out)))
        return out

    @property
    def total_nodes(self):
        """Nodes of all zones concatenated in zone order: the rows of network_check's arrays."""
        return int(sum(n or 0 for n in self.node_counts))

    def network_check(self, source="schedule", vset=1.0, vlow=0.95, vhigh=1.05, row_tol=1e-9, scale=None, full=False,
                      zones=False, out=None):
        """Voltages and line loadings of every node of every zone, per step, in one call (include/revs_admm.h:
        revs_network_check).  source: "schedule" (P_sch of the last ADMM run), "estimate" (P_est), "repaired" (the
        schedule of the last repair_schedule of that run), "central" (the kept schedule of the last central_bracket) or a host
        schedule P [H, T].  scale: [total_nodes] signed 1/rating per edge (None = 1).  Returns dict(summary=dict,
        voltage=[total_nodes, T], loading=[total_nodes, T], zone_worst=[zones, 3]); the arrays are None unless
        asked for with full / zones.  out: optional dict of C-contiguous float64 [total_nodes, T] arrays voltage
        and loading to write into."""
        N, T = self.total_nodes, self.T
        Pp = None
        if isinstance(source, str):
            src = {"schedule": REVS_NET_SCHEDULE, "estimate": REVS_NET_ESTIMATE, "repaired": REVS_NET_REPAIRED,
                   "central": REVS_NET_CENTRAL}.get(source)
            if src is None:
                raise ValueError("source must be 'schedule', 'estimate', 'repaired', 'central' or an [H, T] array, "
                                 f"not {source!r}")
        else:
            src, Pp = REVS_NET_HOST, _f64(source, (self.H, T))
        sc = None if scale is None else _f64(scale, (N,))
        V = L = None
        if full:
            if out is not None:
                V, L = out["voltage"], out["loading"]
                for a in (V, L):
                    if a.shape != (N, T) or a.dtype != np.float64 or not a.flags.c_contiguous:
                        raise ValueError(f"out arrays must be C-contiguous float64 of shape {(N, T)}")
            else:
                V, L = np.empty((N, T)), np.empty((N, T))
        Z = np.empty((self.nf, 3)) if zones else None
        summ = NetworkSummary()
        _check(self.lib.revs_network_check(self._h, src, _dp(Pp), vset, vlow, vhigh, row_tol, _dp(sc), _dp(V), _dp(L),
                                           _dp(Z), C.byref(summ)))
        return dict(summary=summ.as_dict(), voltage=V, loading=L, zone_worst=Z)

    def _schedule_out(self, schedule, mask):
        """The host buffers of a tool's schedule, each None unless asked for: P_sch [H, T] and the charging bits
        [H, ceil(T/64)] uint64, with the (P_out, hour_mask, mask_words) arguments of the library call."""
        W = (self.T + 63) // 64
        P = np.empty((self.H, self.T)) if schedule else None
        M = np.empty((self.H, W), dtype=np.uint64) if mask else None
        return P, M, (_dp(P), None if M is None else M.ctypes.data_as(C.POINTER(C.c_uint64)), W)

    def repair_schedule(self, vset=1.0, vhigh=1.05, row_tol=1e-9, schedule=True, mask=False):
        """Greedy voltage repair of the last ADMM run's charging decisions, zone by zone on the device
        (include/revs_admm.h: revs_repair_schedule; a heuristic, a zone may be left with violated rows).  Returns
        dict(P_sch=[H, T] repaired schedule or None, mask=[H, ceil(T/64)] uint64 charging bits or None,
        zone_info=[zones, 3] int32 {status 0 untouched / 1 repaired / 2 violations left, hours moved, hours dropped},
        moves, drops, zones_violated, zones_repaired, zones_left).  P_sch, P_est and the results of the run stay as
        they are; expand_schedule(mask, ...) gives the repaired P_ev and SOC."""
        P, M, args = self._schedule_out(schedule, mask)
        Z = np.zeros((self.nf, 3), dtype=np.int32)
        _check(self.lib.revs_repair_schedule(self._h, vset, vhigh, row_tol, *args,
                                             Z.ctypes.data_as(C.POINTER(C.c_int32))))
        return repair_totals(dict(P_sch=P, mask=M, zone_info=Z))

    def central_bracket(self, vset=1.0, vhigh=1.05, row_tol=1e-9, iters=100, schedule=True, mask=False):
        """Bracket of the centralized optimum zone by zone on the device (include/revs_admm.h: revs_central_bracket):
        a voltage-feasible binary schedule (UB) and a Lagrangian lower bound (LB) per zone, from the homes, tariff and
        trees alone.  Returns dict(P_sch=[H, T] kept schedule or None, mask=[H, ceil(T/64)] uint64 charging bits or
        None, zone_bounds=[zones, 2] {LB, UB}, zone_info=[zones, 3] int32 {status 0 optimal / 1 bracketed / 2 no
        feasible schedule found / 3 certified infeasible, ascent steps, repair moves + drops of the kept start}) and
        the totals of central_totals.  Nothing of an ADMM run is read or changed."""
        P, M, args = self._schedule_out(schedule, mask)
        B = np.zeros((self.nf, 2))
        Z = np.zeros((self.nf, 3), dtype=np.int32)
        _check(self.lib.revs_central_bracket(self._h, vset, vhigh, row_tol, int(iters), *args, _dp(B),
                                             Z.ctypes.data_as(C.POINTER(C.c_int32))))
        return central_totals(dict(P_sch=P, mask=M, zone_bounds=B, zone_info=Z))

    def certify_infeasible(self, vset, vhigh, row_tol=1e-9):
        """Certificate of voltage infeasibility zone by zone on the device (include/revs_admm.h:
        revs_certify_infeasible): a proof that no binary schedule keeps the SOC windows, plug-in windows and voltage
        rows, from the homes and trees alone.  Returns dict(zone_cert=[zones, 4] int32 {kind 0 no proof / 1 base load /
        2 counting, residence (local), step (kind 1) or k (kind 2), need - cap (kind 2)}) with the counts of
        certify_totals.  Nothing of an ADMM run or of central_bracket is read or changed."""
        Z = np.zeros((self.nf, 4), dtype=np.int32)
        _check(self.lib.revs_certify_infeasible(self._h, vset, vhigh, row_tol, Z.ctypes.data_as(C.POINTER(C.c_int32)),
                                                None))
        return certify_totals(dict(zone_cert=Z))

    def hosting_capacity(self, source="schedule", vset=1.0, vhigh=1.05, row_tol=1e-9, scale=None, homes=True,
                         uniform=True):
        """Hosting capacity of a schedule zone by zone on the device (include/revs_admm.h: revs_hosting_capacity): how
        many more kW every home can draw at every step, with everything else unchanged, before a voltage row
        (R P)_i - (vhigh^2 - vset^2) <= row_tol or a rated line binds.  source as in network_check; scale: [total_nodes]
        signed 1/rating per edge, 0 = unrated (None: no edge is rated).  Returns dict(home_cap=[H, T] kW or None,
        zone_uniform=[zones, T] kW every residence of the zone can add at once, or None, zone_counts=[zones, 3] int64
        {window steps, window steps where one more charger fits, thermally bound (home, step) pairs}) with the totals of
        hosting_totals.  Nothing else is read or changed."""
        T = self.T
        Pp = None
        if isinstance(source, str):
            src = {"schedule": REVS_NET_SCHEDULE, "estimate": REVS_NET_ESTIMATE, "repaired": REVS_NET_REPAIRED,
                   "central": REVS_NET_CENTRAL}.get(source)
            if src is None:
                raise ValueError("source must be 'schedule', 'estimate', 'repaired', 'central' or an [H, T] array, "
                                 f"not {source!r}")
        else:
            src, Pp = REVS_NET_HOST, _f64(source, (self.H, T))
        sc = None if scale is None else _f64(scale, (self.total_nodes,))
        cap = np.empty((self.H, T)) if homes else None
        uni = np.empty((self.nf, T)) if uniform else None
        cnt = np.zeros((self.nf, 3), dtype=np.int64)
        _check(self.lib.revs_hosting_capacity(self._h, src, _dp(Pp), vset, vhigh, row_tol, _dp(sc), _dp(cap), _dp(uni),
                                              cnt.ctypes.data_as(C.POINTER(C.c_int64))))
        return hosting_totals(dict(home_cap=cap, zone_uniform=uni, zone_counts=cnt), self.off)

    # ---- the same check with the rows partitioned over the GPUs of the box; the all-gather of the result is fused
    # into the epilogue of the contraction kernel (peer-memory stores, include/revs_admm.h: revs_gather_*)
    def gather_export(self, capacity_doubles):
        buf = C.create_string_buffer(64)
        _check(self.lib.revs_gather_export(self._h, int(capacity_doubles), buf))
        return buf.raw

    def gather_attach(self, world, rank, handles):
        handles = bytes(handles)
        assert len(handles) == 64 * world
        _check(self.lib.revs_gather_attach(self._h, world, rank, handles))

    def reliability_sharded(self, feeder, kind, rows, P, vset=1.0, scale=None):
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        out = np.empty((len(rows), self.T))
        sc = None if scale is None else _f64(scale, (len(rows),))
        Pp = _f64(P, (self.sizes[feeder], self.T))
        _check(self.lib.revs_reliability_sharded(self._h, feeder, kind, len(rows),
                                                 rows.ctypes.data_as(C.POINTER(C.c_int32)), _dp(sc), vset,
                                                 _dp(Pp), _dp(out)))
        return out

    # ---- residual all-reduce over the GPUs of the box (peer-memory mailboxes, see include/revs_admm.h)
    def comm_export(self):
        buf = C.create_string_buffer(64)
        _check(self.lib.revs_comm_export(self._h, buf))
        return buf.raw

    def comm_attach(self, world, rank, handles):
        handles = bytes(handles)
        assert len(handles) == 64 * world
        _check(self.lib.revs_comm_attach(self._h, world, rank, handles))

    def comm_detach(self):
        _check(self.lib.revs_comm_detach(self._h))

    def set_option(self, name, value):
        _check(self.lib.revs_set_option(self._h, name.encode(), float(value)))

    def stats(self):
        st = Stats()
        _check(self.lib.revs_get_stats(self._h, C.byref(st)))
        return st.as_dict()

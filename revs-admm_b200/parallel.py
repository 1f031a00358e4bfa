"""Multi-GPU driver: one process per B200, feeders sharded across ranks.

The ADMM loop of the reference couples homes only through their own feeder's sensitivity
block (Utility.network, lpsolver.py:183-194, is block-diagonal over feeders), so whole
feeders are the unit of distribution: every rank owns a contiguous, home-balanced slice of
the feeder list and runs the device loop on it.  The only exchange per iteration is the
global convergence test -- three scalars (residual sums and the home-hour count) summed
with one all-reduce (NCCL over NVLink on GPUs, gloo in the CPU tests).  With tol <= 0 (the
reference's fixed iteration count) even that is only needed for reporting.
"""
import os

import numpy as np


def shard_feeders(sizes, world_size, rank):
    """Contiguous slice [lo, hi) of the feeder list for `rank`, balancing homes."""
    sizes = np.asarray(sizes, dtype=np.int64)
    if world_size <= 1:
        return 0, len(sizes)
    cum = np.concatenate([[0], np.cumsum(sizes)])
    total = cum[-1]
    bounds = [int(np.searchsorted(cum, total * r / world_size, side="left")) for r in range(world_size + 1)]
    bounds[0], bounds[-1] = 0, len(sizes)
    for r in range(1, world_size + 1):
        bounds[r] = max(bounds[r], bounds[r - 1])
    return bounds[rank], bounds[rank + 1]


def allreduce_sums(sums, device=None):
    """Sum the per-rank residual sums {sum primal^2, sum dual^2, home-hours} over all ranks."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return np.asarray(sums, dtype=np.float64)
    t = torch.tensor(np.asarray(sums, dtype=np.float64), dtype=torch.float64, device=device or "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t.cpu().numpy()


def attach_peers(solver):
    """Give `solver` (a _cabi.Solver on this rank's GPU) the global stopping rule: exchange the IPC handles of
    the residual mailboxes over torch.distributed and attach them (include/revs_admm.h: revs_comm_*).  From then
    on the all-reduce of the residual sums happens inside the fused dual-update kernel, over NVLink peer memory,
    every iteration -- also inside the captured loop of solve_admm(tol > 0).  No-op for a single rank."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return False
    world, rank = dist.get_world_size(), dist.get_rank()
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    mine = torch.frombuffer(bytearray(solver.comm_export()), dtype=torch.uint8).to(dev)
    got = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(got, mine)
    solver.comm_attach(world, rank, b"".join(bytes(t.cpu().numpy().tobytes()) for t in got))
    dist.barrier()                      # every mailbox is zeroed and mapped before anyone starts a run
    return True


def attach_gather(solver, capacity_doubles):
    """Prepare `solver` for reliability_sharded(): every rank allocates its gather buffer (room for
    `capacity_doubles` = rows x T outputs), the IPC handles travel over torch.distributed, every rank maps every
    buffer.  Afterwards each rank contracts only its block of the rows of a feeder and the contraction kernel
    itself stores the result into all buffers over NVLink (include/revs_admm.h: revs_gather_*).  Single rank:
    the buffer is attached to itself, the call degenerates to the plain check."""
    import torch
    import torch.distributed as dist
    mine_raw = solver.gather_export(capacity_doubles)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        solver.gather_attach(1, 0, mine_raw)
        return 1
    world, rank = dist.get_world_size(), dist.get_rank()
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    mine = torch.frombuffer(bytearray(mine_raw), dtype=torch.uint8).to(dev)
    got = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(got, mine)
    solver.gather_attach(world, rank, b"".join(bytes(t.cpu().numpy().tobytes()) for t in got))
    dist.barrier()                      # every buffer is zeroed and mapped before anyone stores into it
    return world


def row_block(n_rows, tile_rows, world, rank):
    """Rows [lo, hi) of a row-partitioned contraction that rank `rank` of `world` owns: contiguous blocks of whole
    tiles (csrc/revs_capi.cu: reliability_impl uses the same rule)."""
    tiles = (n_rows + tile_rows - 1) // tile_rows
    lo = min(n_rows, (tiles * rank // world) * tile_rows)
    hi = min(n_rows, (tiles * (rank + 1) // world) * tile_rows)
    return lo, hi


def residuals(total_sums, kappa):
    sp, sd, cnt = total_sums
    return float(np.sqrt(sp / cnt)), float(kappa * np.sqrt(sd / cnt))


def run_admm(stepper, kappa=5.0, iter_max=15, vset=1.0, vlow=0.95, vhigh=1.05, tol=0.0, device=None, global_sums=False):
    """Drive `stepper` (a _cabi.Solver, or anything with admm_begin/admm_step) for this
    rank's feeders one iteration at a time; stop on the GLOBAL residuals.  Returns (iterations, history).
    ``global_sums``: the stepper's sums already run over all ranks (attach_peers), no host all-reduce.
    (The fast path is ``attach_peers(solver); solver.solve_admm(tol=...)``: one captured loop per rank.)"""
    stepper.admm_begin(kappa=kappa, iter_max=iter_max, vset=vset, vlow=vlow, vhigh=vhigh)
    history = []
    for k in range(iter_max):
        local = stepper.admm_step()
        if tol > 0.0:
            r, s = residuals(local if global_sums else allreduce_sums(local, device), kappa)
            history.append((r, s))
            if r < tol and s < tol:
                return k + 1, history
        else:
            history.append(tuple(local[:2]))
    return iter_max, history


# maxima of a network-check summary: value, zone, (index, step) and the fields that travel with the value
_NET_MAXIMA = (("drop_max", "drop_zone", "drop_node", "drop_step", ("v_min",)),
               ("row_excess_max", "excess_zone", "excess_res", "excess_step", ()),
               ("loading_max", "loading_zone", "loading_node", "loading_step", ()))
_NET_COUNTS = ("rows_violated", "nodes_below_vlow", "edges_overloaded")


def merge_network_summaries(summaries, zone_offsets):
    """One network-check summary (Solver.network_check()["summary"]) from those of solvers that hold consecutive
    blocks of the zones: part k's zone z is zone zone_offsets[k] + z of the whole.  The rule of the library: every
    maximum goes to the largest value, ties to the lowest (zone, index, step); a part without a candidate (zone -1,
    e.g. no residence) is skipped; counts are summed."""
    out = dict(summaries[0])
    for key in _NET_COUNTS:
        out[key] = int(sum(int(s[key]) for s in summaries))
    for val, zk, ik, tk, extra in _NET_MAXIMA:
        best, win = None, None
        for s, z0 in zip(summaries, zone_offsets):
            if s[zk] < 0:
                continue
            key = (s[val], int(z0) + s[zk], s[ik], s[tk])
            if best is None or key[0] > best[0] or (key[0] == best[0] and key[1:] < best[1:]):
                best, win = key, s
        if best is None:
            out.update({val: -np.inf, zk: -1, ik: -1, tk: -1})
        else:
            out.update({val: best[0], zk: best[1], ik: best[2], tk: best[3]})
            out.update({e: win[e] for e in extra})
    return out


def _pinned_empty(shape):
    """Page-locked host scratch (torch is only the allocator); plain numpy if torch has no CUDA."""
    try:
        import torch
        if torch.cuda.is_available():
            t = torch.empty(tuple(shape), dtype=torch.float64).pin_memory()
            return t.numpy(), t
    except Exception:
        pass
    return np.empty(shape), None


class PipelinedSolver:
    """Several independent solver pipelines on ONE GPU.

    The sensitivity matrix is block diagonal over voltage zones, so a GPU's zones can be cut into
    K contiguous groups that never exchange data.  Each group gets its own device solver (own
    streams, own working-set state) and its own host thread; while one pipeline sits in the
    latency-bound tail of a utility solve or in a host round trip, the others keep the SMs busy.
    Same methods as ``_cabi.Solver``; results are those of a single solver, bit for bit.
    """

    def __init__(self, feeder_sizes, T, device=0, pipelines=4):
        from concurrent.futures import ThreadPoolExecutor
        from ._cabi import Solver
        self.sizes = [int(n) for n in feeder_sizes]
        self.T, self.nf = int(T), len(self.sizes)
        self.off = np.concatenate([[0], np.cumsum(self.sizes)]).astype(np.int64)
        self.H = int(self.off[-1])
        K = max(1, min(int(pipelines), self.nf))
        self.cuts = [shard_feeders(self.sizes, K, k) for k in range(K)]
        self.cuts = [(a, b) for a, b in self.cuts if b > a]
        self.parts = [Solver(self.sizes[a:b], T, device=device) for a, b in self.cuts]
        self.rows = [(int(self.off[a]), int(self.off[b])) for a, b in self.cuts]
        self.pool = ThreadPoolExecutor(max_workers=len(self.parts))
        self._diff_scratch = {}
        # Stream priorities: the first pipeline one level above the others.  It is the first to have its inputs on
        # the device in schedule(), finishes ~2 ms before the rest, and its download overlaps their compute (end to end
        # 15.2 -> 14.8 ms on the bench population; the device-resident time does not change).  Measured without gain:
        # every pipeline on its own level, or any other pipeline favoured (profiles/README_r02.md).
        # REVS_PIPELINE_PRIORITY=0 switches it off, =1 puts every pipeline on its own level.
        mode = os.environ.get("REVS_PIPELINE_PRIORITY", "first")
        if len(self.parts) > 1 and mode != "0":
            for k, p in enumerate(self.parts):
                p.set_option("priority", k if mode == "1" else min(k, 1))

    # ---- plumbing
    def _diff_buf(self, k, iters):
        """Page-locked [iters, homes of pipeline k] buffer for the per-iteration convergence values
        (a column slice of the caller's [iters, H] array is not contiguous)."""
        lo, hi = self.rows[k]
        key = (k, iters)
        if key not in self._diff_scratch:
            self._diff_scratch[key] = _pinned_empty((iters, hi - lo))
        return self._diff_scratch[key][0]

    def _each(self, fn, concurrent=True):
        if concurrent and len(self.parts) > 1:
            return list(self.pool.map(fn, range(len(self.parts))))
        return [fn(k) for k in range(len(self.parts))]

    def close(self):
        for p in getattr(self, "parts", []):
            p.close()
        self.parts = []
        if getattr(self, "pool", None):
            self.pool.shutdown(wait=True)
            self.pool = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- inputs
    def set_feeder_trees(self, trees):
        assert len(trees) == self.nf
        self._each(lambda k: self.parts[k].set_feeder_trees(trees[self.cuts[k][0]:self.cuts[k][1]]))

    def set_homes(self, **hm):
        def f(k):
            lo, hi = self.rows[k]
            self.parts[k].set_homes(**{n: v[lo:hi] for n, v in hm.items()})
        self._each(f)

    def set_tariff(self, cost):
        self._each(lambda k: self.parts[k].set_tariff(cost), concurrent=False)

    def set_option(self, name, value):
        self._each(lambda k: self.parts[k].set_option(name, value), concurrent=False)

    # ---- solves
    def solve_admm(self, concurrent=True, **kw):
        """tol <= 0 (the reference's fixed iteration count): every pipeline runs its whole captured loop on its
        own.  tol > 0: the stopping rule is GLOBAL (both residuals over all homes below tol), so the pipelines
        advance in lock-step, one iteration at a time, and their residual sums are combined between steps --
        every pipeline runs the same number of iterations and the result is that of a single solver."""
        tol = float(kw.get("tol", 0.0) or 0.0)
        if tol <= 0.0 or len(self.parts) == 1:
            return max(self._each(lambda k: self.parts[k].solve_admm(**kw), concurrent=concurrent))
        kw = {k: v for k, v in kw.items() if k != "tol"}
        kappa, iter_max = float(kw.get("kappa", 5.0)), int(kw.get("iter_max", 15))
        self._each(lambda k: self.parts[k].admm_begin(**kw), concurrent=concurrent)
        for it in range(iter_max):
            sums = np.sum(self._each(lambda k: self.parts[k].admm_step(), concurrent=concurrent), axis=0)
            r, s_ = residuals(sums, kappa)
            if r < tol and s_ < tol:
                return it + 1
        return iter_max

    def schedule(self, trees, homes, cost, out=None, compact=False, **admm):
        """Host buffers in, host results out -- the whole path of lpsolver.solve_ADMM for this GPU's
        zones.  Every pipeline runs upload -> solve -> download on its own thread.  The host-side
        preparation of the uploads (padded layouts, cumulative resistances) runs concurrently; the
        copies themselves take the PCIe link one pipeline at a time (a per-device lock inside the
        library), so a pipeline starts computing while the next one is still uploading, and the
        downloads of the pipelines that finish first overlap the compute of the others.
        ``compact``: results come back as P_sch + charging bit masks + diff (Solver.schedule_compact;
        _cabi.expand_schedule rebuilds P_ev / SOC on request) -- a third of the D2H bytes."""
        import threading
        import time
        if float(admm.get("tol", 0.0) or 0.0) > 0.0 and len(self.parts) > 1:
            raise ValueError("schedule() overlaps whole pipelines and cannot apply a global stopping rule; "
                             "use the set_* calls and solve_admm(tol=...) (lock-step) instead")
        H, T = self.H, self.T
        iters = int(admm.get("iter_max", 15))
        if out is None:
            out = dict(P_sch=np.empty((H, T)), diff=np.empty((iters, H)))
            if compact:
                out["mask"] = np.empty((H, (T + 63) // 64), dtype=np.uint64)
            else:
                out.update(P_ev=np.empty((H, T)), SOC=np.empty((H, T + 1)))
        D = out.get("diff")
        d2h = threading.Lock()
        prep = [threading.Event() for _ in range(len(self.parts) + 1)]
        prep[0].set()
        trace = os.environ.get("REVS_DEBUG_E2E") is not None
        t_origin = time.perf_counter()
        marks = [None] * len(self.parts)

        def f(k):
            lo, hi = self.rows[k]
            a, b = self.cuts[k]
            tm = [time.perf_counter()]
            # the interpreter-side packing of the zone arrays holds the GIL: pipeline by pipeline, in order, so that
            # the first pipeline reaches the library (which releases it) as early as possible
            prep[k].wait()
            try:
                packed = self.parts[k].pack_trees(trees[a:b])
            finally:
                prep[k + 1].set()
            self.parts[k].set_feeder_trees(None, packed=packed)
            tm.append(time.perf_counter())
            self.parts[k].set_homes(**{n: v[lo:hi] for n, v in homes.items()})
            self.parts[k].set_tariff(cost)
            tm.append(time.perf_counter())
            done = self.parts[k].solve_admm(**admm)
            tm.append(time.perf_counter())
            with d2h:
                tm.append(time.perf_counter())
                if compact:
                    # the convergence values go straight into this pipeline's column block of the caller's array
                    sub = dict(P_sch=out["P_sch"][lo:hi], mask=out["mask"][lo:hi], diff=None if D is None else D[:, lo:hi])
                    self.parts[k].schedule_compact(want_diff=D is not None, out=sub)
                else:
                    sub = dict(P_sch=out["P_sch"][lo:hi], P_ev=out["P_ev"][lo:hi], SOC=out["SOC"][lo:hi],
                               diff=self._diff_buf(k, iters) if D is not None else None)
                    self.parts[k].results(iters, want_diff=D is not None, out=sub)
            tm.append(time.perf_counter())
            if D is not None and not compact:
                D[:done, lo:hi] = sub["diff"][:done]
            tm.append(time.perf_counter())
            marks[k] = tm
            return done
        self._each(f)
        if trace:
            import sys
            for k, tm in enumerate(marks):
                print("[revs e2e] pipeline %d: " % k + "  ".join(
                    "%s %.2f" % (n, 1e3 * (t - t_origin)) for n, t in zip(
                        ("start", "trees", "homes", "solved", "d2h-lock", "downloaded", "done"), tm)), file=sys.stderr, flush=True)
        out["diff"] = D
        return out

    def results(self, iters=None, want_diff=True, out=None):
        H, T = self.H, self.T
        done = [p.stats()["admm_iterations"] for p in self.parts]      # equal: fixed count, or lock-step under tol > 0
        iters = max(done) if iters is None else max(iters, max(done))
        if out is None:
            out = dict(P_sch=np.empty((H, T)), P_ev=np.empty((H, T)), SOC=np.empty((H, T + 1)),
                       diff=np.zeros((iters, H)) if want_diff else None)
        D = out.get("diff")
        if D is not None and D.shape[0] < max(done):
            raise ValueError(f"out['diff'] has {D.shape[0]} rows but {max(done)} iterations ran")

        def f(k):
            lo, hi = self.rows[k]
            sub = dict(P_sch=out["P_sch"][lo:hi], P_ev=out["P_ev"][lo:hi], SOC=out["SOC"][lo:hi],
                       diff=self._diff_buf(k, iters) if D is not None else None)
            self.parts[k].results(iters, want_diff=D is not None, out=sub)       # the library checks the row capacity
            if D is not None:
                D[:done[k], lo:hi] = sub["diff"][:done[k]]
        self._each(f)
        return dict(P_sch=out["P_sch"], P_ev=out["P_ev"], SOC=out["SOC"], diff=D)

    def estimate(self):
        pe, gm = np.empty((self.H, self.T)), np.empty((self.H, self.T))

        def f(k):
            lo, hi = self.rows[k]
            pe[lo:hi], gm[lo:hi] = self.parts[k].estimate()
        self._each(f)
        return pe, gm

    def network_check(self, source="schedule", scale=None, full=False, zones=False, **kw):
        """Solver.network_check over all pipelines at once: every pipeline checks its zones concurrently and writes
        its contiguous block of nodes into the [total nodes, T] arrays; the summaries are merged with the zones
        numbered over the whole population (merge_network_summaries), zone_worst is concatenated in zone order.
        The result is that of a single solver, bit for bit."""
        node_off = np.concatenate([[0], np.cumsum([p.total_nodes for p in self.parts])]).astype(np.int64)
        N, T = int(node_off[-1]), self.T
        host = not isinstance(source, str)
        if host:
            source = np.ascontiguousarray(source, dtype=np.float64)
            if source.shape != (self.H, T):
                raise ValueError(f"expected shape {(self.H, T)}, got {source.shape}")
        if scale is not None:
            scale = np.ascontiguousarray(scale, dtype=np.float64)
            if scale.shape != (N,):
                raise ValueError(f"expected shape {(N,)}, got {scale.shape}")
        out = dict(voltage=np.empty((N, T)), loading=np.empty((N, T))) if full else None

        def f(k):
            lo, hi = self.rows[k]
            a, b = node_off[k], node_off[k + 1]
            return self.parts[k].network_check(source=source[lo:hi] if host else source,
                                               scale=None if scale is None else scale[a:b], full=full, zones=zones,
                                               out=None if out is None else {n: v[a:b] for n, v in out.items()}, **kw)
        res = self._each(f)
        return dict(summary=merge_network_summaries([r["summary"] for r in res], [a for a, _ in self.cuts]),
                    voltage=None if out is None else out["voltage"], loading=None if out is None else out["loading"],
                    zone_worst=np.concatenate([r["zone_worst"] for r in res]) if zones else None)

    def _zone_order(self, method, totals, *args, part_kw=None, **kw):
        """Solver.<method> on every pipeline at once: each array of the results concatenated in zone order (None where
        not asked for) and the totals recomputed by `totals` -- the bytes of a single solver over the same zones.
        part_kw(k): optional further keyword arguments of pipeline k (its share of a per-home or per-node input)."""
        res = self._each(lambda k: getattr(self.parts[k], method)(*args, **kw, **(part_kw(k) if part_kw else {})))
        return totals({n: None if v is None else np.concatenate([r[n] for r in res])
                       for n, v in res[0].items() if v is None or isinstance(v, np.ndarray)})

    def repair_schedule(self, schedule=True, mask=False, **kw):
        """Solver.repair_schedule over all pipelines at once (_zone_order)."""
        from ._cabi import repair_totals
        return self._zone_order("repair_schedule", repair_totals, schedule=schedule, mask=mask, **kw)

    def central_bracket(self, schedule=True, mask=False, **kw):
        """Solver.central_bracket over all pipelines at once (_zone_order)."""
        from ._cabi import central_totals
        return self._zone_order("central_bracket", central_totals, schedule=schedule, mask=mask, **kw)

    def certify_infeasible(self, *args, **kw):
        """Solver.certify_infeasible over all pipelines at once (_zone_order)."""
        from ._cabi import certify_totals
        return self._zone_order("certify_infeasible", certify_totals, *args, **kw)

    def hosting_capacity(self, source="schedule", scale=None, homes=True, uniform=True, **kw):
        """Solver.hosting_capacity over all pipelines at once (_zone_order); a host schedule [H, T] and scale
        [total nodes] are cut into every pipeline's rows of homes and nodes."""
        from ._cabi import hosting_totals
        node_off = np.concatenate([[0], np.cumsum([p.total_nodes for p in self.parts])]).astype(np.int64)
        host = not isinstance(source, str)
        if host:
            source = np.ascontiguousarray(source, dtype=np.float64)
            if source.shape != (self.H, self.T):
                raise ValueError(f"expected shape {(self.H, self.T)}, got {source.shape}")
        if scale is not None:
            scale = np.ascontiguousarray(scale, dtype=np.float64)
            if scale.shape != (int(node_off[-1]),):
                raise ValueError(f"expected shape {(int(node_off[-1]),)}, got {scale.shape}")

        def part(k):
            (lo, hi), a, b = self.rows[k], node_off[k], node_off[k + 1]
            return dict(source=source[lo:hi] if host else source, scale=None if scale is None else scale[a:b])
        return self._zone_order("hosting_capacity", lambda r: hosting_totals(r, self.off), part_kw=part, homes=homes,
                                uniform=uniform, **kw)

    def stats(self):
        """Counters and CUDA-event spans summed over the pipelines; total_ms is the longest
        pipeline (they run side by side), residuals are recombined from the per-pipeline norms."""
        sts = [p.stats() for p in self.parts]
        out = {}
        for key in sts[0]:
            vals = [s[key] for s in sts]
            if key in ("total_ms", "admm_iterations", "max_working_set"):
                out[key] = max(vals)
            elif key in ("primal_residual", "dual_residual"):
                w = [hi - lo for lo, hi in self.rows]
                out[key] = float(np.sqrt(sum(v * v * n for v, n in zip(vals, w)) / max(sum(w), 1)))
            else:
                out[key] = sum(vals)
        out["total_ms_sum"] = sum(s["total_ms"] for s in sts)
        out["pipelines"] = len(sts)
        return out

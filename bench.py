#!/usr/bin/env python
"""REVS ADMM benchmark (driver contract: one JSON line on stdout from rank 0).

A "step" is one complete distributed-ADMM schedule (reference: lpsolver.solve_ADMM,
max_iterations = 15 as in revs_config.yaml) of this rank's synthetic home population:
weak scaling, 125k homes x 96 quarter-hour steps per GPU in feeders of 1000 residences
(8 GPUs = the 1M-home target of BASELINE.json).  metric = home-hours scheduled per second
(homes x 24 h of horizon / time of the whole schedule, all ranks).

  value : device-resident inputs, timed with CUDA events on the library's own stream
  e2e   : the C-ABI call sequence a reference user makes, HOST buffers in, HOST results out
          (set_feeder_tree, set_homes, set_tariff, solve_admm, get_results) inside the
          timed region
  roofline / kernels : per-kernel achieved rates from the library's CUDA-event spans
  cpu_baseline : the CPU oracle (a port of the reference: Gurobi is not installable) on a
          bounded sample of the same workload, host cores of this box, rank 0 / N=1 only

`--impl reference` times that CPU port as the reference arm.
`--dump-outputs DIR` writes the results of the last timed step of `value` as .npy files (dump_outputs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HOURS = 24.0
WORKLOADS = {
    # name: (population of revs_admm_b200/feeder.py:POPULATIONS, feeders per GPU)
    "synthetic-refshape-125k-homes-per-gpu-x96": ("refshape", 125),      # zones of 149..297 residences, voltage-feasible base load
    "synthetic-multifeeder-125k-homes-per-gpu-x96": ("laterals", 125),   # round-1 population: zones of 43..165, base load over the limit
    "synthetic-radial-10k-homes-x96": ("radial10k", 1),                  # BASELINE.json config 3: one dense 10k x 10k zone
    "synthetic-refshape-100k-homes-x96": ("refshape", 100),              # BASELINE.json config 4 (strong scaling over 2/4/8 GPUs)
    "tiny": ("refshape", 1),
}
ADMM = dict(kappa=5.0, iter_max=15, vset=1.03, vlow=0.95, vhigh=1.05)   # revs_config.yaml / revs_fixture.py:255-259
DUMP_HOMES = 8192     # homes (rows) written by --dump-outputs: 33 MB of float64 at the workloads' T = 96, kept below 64 MB


def workload_shape(workload):
    """(feeders per GPU, homes per feeder, T) of a workload."""
    from revs_admm_b200.feeder import POPULATIONS
    pop, nf = WORKLOADS[workload]
    return nf, POPULATIONS[pop]["homes"], POPULATIONS[pop]["T"]


def make_rank_problem(workload, rank, split=True, strong=None):
    """Synthetic feeders + homes of this rank.  Every rank draws ITS OWN population (seed = rank;
    REVS_BENCH_SEED=<int> pins one draw for all ranks).  With `split` every feeder is handed to the
    solver as its independent voltage zones.  `strong` = (world, rank): the workload's feeders are
    one fixed population cut into `world` contiguous shares (strong scaling)."""
    from revs_admm_b200.feeder import population
    pop, nf = WORKLOADS[workload]
    seed_env = os.environ.get("REVS_BENCH_SEED", "rank")
    if strong is not None:
        world, r = strong
        lo, hi = nf * r // world, nf * (r + 1) // world
        return population(pop, hi - lo, seed=0 if seed_env == "rank" else int(seed_env), split=split, first_feeder=lo)
    seed = rank if seed_env == "rank" else int(seed_env)
    return population(pop, nf, seed=seed, split=split)


def pinned_like(a):
    """Copy into page-locked host memory (torch is only the allocator here)."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t.numpy(), t


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region (NVML every 20 ms; nvidia-smi as fallback)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.th = threading.Thread(target=self._run, daemon=True)
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _run(self):
        nv = self.nvml
        while not self.stop.is_set():
            try:
                if nv is not None:
                    sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                        else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    flags = ["Active" if r & m else "Not Active" for m in (0x8, 0x40, 0x20, 0x4)]  # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
                    self.rows.append([str(sm), str(self.max_sm), "0"] + flags)
                    self.stop.wait(0.02)
                    continue
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def dump_outputs(path, s):
    """Write what the caller of the timed path receives after its last step -- the schedule (Solver.results) and
    the operator's estimate and multipliers (Solver.estimate) -- as float64 DIR/<name>.npy, so that two builds can be
    compared output for output.  Populations above DUMP_HOMES homes are sampled: the same seeded set of homes every
    run, listed in home_index.npy."""
    res = s.results()
    res["P_est"], res["Gamma"] = s.estimate()
    H = s.H
    rows = np.arange(H) if H <= DUMP_HOMES else np.sort(np.random.default_rng(0).choice(H, DUMP_HOMES, replace=False))
    arrays = {k: (v[:, rows] if k == "diff" else v[rows]) for k, v in res.items()}     # diff is [iterations, homes]
    arrays["home_index"] = rows
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def fp64_gemm_peak_tflops():
    """cuBLAS DGEMM on this box: the denominator for the FP64 tensor-core contraction
    (MEASURED_PEAKS.json has no fp64 figure)."""
    import torch
    n = 6144
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


# ------------------------------------------------------------------------------ CPU reference arm
def _cpu_feeder_job(job):
    """One feeder of the workload through the CPU oracle (runs in a worker process, BLAS single-threaded)."""
    workload, first, no_split, iters, one_thread = job
    if one_thread:                                   # one feeder per worker process: BLAS single-threaded inside
        try:
            from threadpoolctl import threadpool_limits
            threadpool_limits(limits=1)
        except Exception:
            pass
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import revs_oracle as O
    from revs_admm_b200.feeder import population
    pop, _ = WORKLOADS[workload]
    trees, hm, cost, sizes, T = population(pop, 1, seed=0, split=not no_split, first_feeder=first)
    Rb = [O.rmat_from_tree(z.parent, z.r)[np.ix_(z.res_node, z.res_node)] for z in trees]
    t0 = time.perf_counter()
    O.solve_ADMM_arrays(Rb, load=hm["load"], cost=cost, ev_mask=hm["has_ev"].astype(bool),
                        rating=hm["rating"], capacity=hm["capacity"], initial=hm["initial"],
                        start=hm["start"], end=hm["end"], **dict(ADMM, iter_max=iters))
    return sum(sizes), time.perf_counter() - t0


def cpu_port_sample(workload, n_feeders=None, no_split=False, workers=None):
    """A bounded sample of the workload through the CPU oracle with ALL host cores: the first
    `n_feeders` feeders of the workload's population (the same feeders the GPU arm's rank 0 holds),
    one worker process per core, feeders dealt to the workers (the ADMM loop is independent per
    feeder), full horizon, all 15 ADMM iterations.  Returns (home_hours/s, seconds, description)."""
    import multiprocessing as mp
    nf, n, T = workload_shape(workload)
    cores = os.cpu_count() or 1
    workers = workers or cores
    k = min(nf, n_feeders or 4 * workers)
    # one big zone (BASELINE.json config 3): the dense port needs minutes per iteration, so the sample is the first 3 of the
    # 15 iterations (BLAS on all cores) and the rate is scaled by 3/15
    iters = ADMM["iter_max"] if n <= 4000 else 3
    jobs = [(workload, f, no_split, iters, workers > 1 and k > 1) for f in range(k)]
    t0 = time.perf_counter()
    if workers > 1 and k > 1:
        with mp.get_context("fork").Pool(min(workers, k)) as pool:
            res = pool.map(_cpu_feeder_job, jobs, chunksize=1)
    else:
        res = [_cpu_feeder_job(j) for j in jobs]
    dt = time.perf_counter() - t0
    homes = sum(r[0] for r in res)
    part = iters / ADMM["iter_max"]
    return homes * HOURS * part / dt, dt, (f"first {k} of {nf} feeders x {n} homes x {T} steps x {iters} of {ADMM['iter_max']} ADMM iterations "
                                           f"(oracle/revs_oracle.py, numpy), {min(workers, k)} worker processes on {cores} cores; "
                                           f"sum of per-feeder CPU seconds {sum(r[1] for r in res):.1f}")


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    vals, secs, desc = [], [], ""
    for i in range(args.warmup + args.steps):
        v, dt, desc = cpu_port_sample(args.workload, args.cpu_sample_feeders)
        if i >= args.warmup:
            vals.append(v)
            secs.append(dt)
    value = float(np.mean(vals))
    nf, n, T = workload_shape(args.workload)
    line = {
        "impl": "reference", "metric": "home_hours_scheduled_per_sec", "value": value, "unit": "home-hours/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(secs)),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "feeders_per_gpu": nf, "homes_per_feeder": n, "T": T, **ADMM},
        "cpu_baseline": {"value": value, "unit": "home-hours/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": "home-hours/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference needs gurobipy (absent, not installable offline); this arm times the CPU port of its algorithm",
    }
    print(json.dumps(line), flush=True)



def objective_check(trees, hm, cost, P_sch, T, sample_zones=64):
    """Centralized-vs-distributed cross-check without a MILP solver (the reference's solve_central,
    lpsolver.py:463-502, minimises sum_h tariff . g_h under the SOC and voltage rows).  A rigorous
    sandwich:  cost of the cheapest SOC-feasible schedule of every home WITHOUT voltage limits
    <= centralized optimum <= cost of the distributed schedule wherever that is voltage-feasible.
    Returns this rank's sums; the voltage check runs on the host over a sample of zones."""
    cost = np.asarray(cost)
    load_cost = float((hm["load"] @ cost).sum())
    ev = hm["has_ev"] > 0
    tt = np.arange(T)[None, :]
    inwin = (tt >= hm["start"][:, None]) & (tt < hm["end"][:, None]) & ev[:, None]
    step = np.where(ev, hm["rating"] / np.maximum(hm["capacity"], 1e-300), 1.0)
    nmin = np.where(ev, np.maximum(np.ceil((0.9 - hm["initial"]) / step - 1e-9), 0), 0).astype(int)
    keyed = np.where(inwin, cost[None, :], np.inf)
    keyed.sort(axis=1)
    csum = np.concatenate([np.zeros((len(keyed), 1)), np.cumsum(np.where(np.isfinite(keyed), keyed, 0.0), axis=1)], axis=1)
    lb = load_cost + float((hm["rating"] * csum[np.arange(len(keyed)), np.minimum(nmin, T)])[ev].sum())
    dist_cost = float((P_sch @ cost).sum())
    u = ADMM["vhigh"] ** 2 - ADMM["vset"] ** 2
    worst, off = -np.inf, 0
    for z, tr in enumerate(trees):
        n = tr.n_res
        if z < sample_zones:
            worst = max(worst, float((tr.drop(P_sch[off:off + n]) - u).max()))      # R_res @ P_sch on the tree, no dense matrix
        off += n
    return dist_cost, lb, worst

# ------------------------------------------------------------------------------ GPU arm
def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import revs_admm_b200 as R
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    try:    # host threads and page-locked buffers next to this rank's GPU (NUMA): matters for the e2e leg at N > 1
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(phys))
    except Exception:
        pass
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    strong = args.scaling == "strong"
    trees, hm, cost, sizes, T = make_rank_problem(args.workload, rank, split=not args.no_split,
                                                  strong=(world, rank) if strong else None)
    H = sum(sizes)
    # page-locked host copies of everything that crosses PCIe in the e2e leg
    keep = []
    hm_p = {}
    for k, v in hm.items():
        hm_p[k], t = pinned_like(v)
        keep.append(t)
    cost_p, t = pinned_like(cost)
    keep.append(t)

    # K independent stream pipelines on this GPU (zones never exchange data): see parallel.PipelinedSolver
    s = R.PipelinedSolver(sizes, T, device=local_rank, pipelines=args.pipelines)

    # results of the end-to-end leg in compact form: the schedule, the charging decisions as bit masks, the convergence
    # values -- P_ev and SOC follow from the masks (revs_admm_b200.expand_schedule, checked below)
    out_p = {}
    for k, shape, dt in (("P_sch", (H, T), np.float64), ("mask", (H, (T + 63) // 64), np.uint64), ("diff", (ADMM["iter_max"], H), np.float64)):
        out_p[k], t = pinned_like(np.empty(shape, dtype=dt))
        keep.append(t)

    def upload():
        s.set_feeder_trees(trees)
        s.set_homes(**hm_p)
        s.set_tariff(cost_p)

    upload()
    stats_acc = {k: 0.0 for k in ("gemm_ms", "gemm_full_ms", "gemm_full_launches", "home_ms", "dual_ms", "qp_ms", "qp_big_ms", "qp_warp_ms", "qp_init_ms", "qp_columns", "qp_warp_rounds", "qp_flops", "total_ms", "total_ms_sum", "kernel_launches",
                                  "gemm_launches", "qp_outer_iterations", "qp_newton_iterations")}
    # ---- device-resident leg ("value")
    for _ in range(args.warmup):
        s.solve_admm(**ADMM)
    barrier()
    with ClockSampler(local_rank) as clk:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dev_ms = 0.0
        host_ms = 0.0
        for _ in range(args.steps):
            th = time.perf_counter()
            s.solve_admm(**ADMM)
            host_ms += (time.perf_counter() - th) * 1e3
            st = s.stats()
            dev_ms += st["total_ms"]
            for k in stats_acc:
                stats_acc[k] += st[k]
        e1.record()
        barrier()
        wall_ms = e0.elapsed_time(e1)
    ms_step = max_over_ranks(wall_ms / args.steps)
    per_rank = [[wall_ms / args.steps, host_ms / args.steps, dev_ms / args.steps]]
    if world > 1:
        tg = [torch.zeros(3, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(tg, torch.tensor(per_rank[0], dtype=torch.float64, device=dev))
        per_rank = [[round(float(x), 3) for x in t.tolist()] for t in tg]
    total_homes = sum_over_ranks(H)
    value = total_homes * HOURS / (ms_step * 1e-3)
    last = s.stats()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, s)

    # ---- end-to-end leg: host buffers in, host results out, every step
    for _ in range(min(args.warmup, 1)):
        s.schedule(trees, hm_p, cost_p, out=out_p, compact=True, **ADMM)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        # one call: feeder trees, homes and tariff up from pinned host buffers, solve, results back to pinned host buffers
        out = s.schedule(trees, hm_p, cost_p, out=out_p, compact=True, **ADMM)
    torch.cuda.synchronize()
    e2e_wall = (time.perf_counter() - t0) * 1e3 / args.steps
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(max(e2e_wall, e0.elapsed_time(e1) / args.steps))
    e2e_value = total_homes * HOURS / (e2e_ms * 1e-3)
    h2d = sum(v.nbytes for v in hm_p.values()) + cost_p.nbytes + sum(tr.parent.nbytes + tr.r.nbytes + tr.res_node.nbytes for tr in trees)
    d2h = sum(v.nbytes for v in out.values() if v is not None)

    # ---- centralized-vs-distributed objective cross-check on the schedule of the last e2e step
    oc_dist, oc_lb, oc_viol = objective_check(trees, hm, cost, out["P_sch"], T)
    oc_dist, oc_lb = sum_over_ranks(oc_dist), sum_over_ranks(oc_lb)
    oc_viol = max_over_ranks(oc_viol)

    # the compact results carry everything revs_get_results returns: rebuild P_ev / SOC from the masks once and compare
    # with the full download of one pipeline's share (outside the timed region)
    compact_ok = None
    if rank == 0:
        lo, hi = s.rows[0]
        full = s.parts[0].results()
        p_ev, soc = R.expand_schedule(out["mask"][lo:hi], T, hm["has_ev"][lo:hi], hm["rating"][lo:hi], hm["capacity"][lo:hi], hm["initial"][lo:hi])
        compact_ok = bool(np.array_equal(p_ev, full["P_ev"]) and np.array_equal(soc, full["SOC"]) and
                          np.array_equal(out["P_sch"][lo:hi], full["P_sch"]))

    # ---- "to convergence": the same population with the stopping rule on (both ADMM residuals below tol), up to
    # conv_iter_max iterations, ONE captured loop per GPU.  With N > 1 the residual sums are all-reduced over the GPUs
    # every iteration inside dual_update_kernel (peer-memory mailboxes over NVLink, revs_comm_*): the collective is in
    # the timed region.  The reference's algorithm is ADMM on a MIQP (binary chargers): where voltage rows bind it
    # settles into a limit cycle of a few homes and the residuals plateau -- `reached` says which.
    conv = None
    if not args.no_convergence:
        sc = R.Solver(sizes, T, device=local_rank)
        sc.set_feeder_trees(trees)
        sc.set_homes(**hm_p)
        sc.set_tariff(cost_p)
        from revs_admm_b200.parallel import attach_peers
        peers = attach_peers(sc) if world > 1 else False
        kwc = dict(ADMM, iter_max=args.conv_iter_max, tol=args.tol)
        sc.solve_admm(**kwc)                       # warm-up: captures the loop for these parameters
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        done = sc.solve_admm(**kwc)
        e1.record()
        barrier()
        cms = max_over_ranks(e0.elapsed_time(e1))
        stc = sc.stats()
        its_all = [done]
        if world > 1:
            tg = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
            dist.all_gather(tg, torch.tensor([done], dtype=torch.int64, device=dev))
            its_all = [int(t.item()) for t in tg]
        # residual trajectory (one more run, stepped, outside the timed region): global sums when peers are attached
        sc.admm_begin(**ADMM | dict(iter_max=args.conv_iter_max))
        traj = []
        for k in range(min(done, args.conv_iter_max)):
            sums = sc.admm_step()
            if k in (0, 1, 2, 4, 9, 14, 24, 49, 99) or k == done - 1:
                traj.append([k + 1, float(np.sqrt(sums[0] / sums[2])), float(ADMM["kappa"] * np.sqrt(sums[1] / sums[2]))])
        conv = {"tol": args.tol, "iter_max": args.conv_iter_max, "iterations": done, "iterations_per_rank": its_all,
                "reached": bool(done < args.conv_iter_max or (stc["primal_residual"] < args.tol and stc["dual_residual"] < args.tol)),
                "ms": cms, "value": total_homes * HOURS / (cms * 1e-3), "unit": "home-hours/s to the stopping rule",
                "admm_iters_per_sec": done / (cms * 1e-3),
                "final_residuals": {"primal": stc["primal_residual"], "dual": stc["dual_residual"]},
                "residual_trajectory [iteration, primal, dual]": traj,
                "allreduce": ("residual sums all-reduced every iteration inside dual_update_kernel over NVLink peer memory, "
                              "%d ranks, inside the timed region" % world) if peers else "single GPU: no exchange",
                "note": "ADMM on a MIQP (binary chargers): with binding voltage rows the reference's iteration ends in a limit cycle; "
                        "reached=false reports the plateau"}
        sc.close()

    # ---- per-kernel achieved rates: one extra single-pipeline solver over all zones of this GPU, host-driven loop
    # (CUDA-event spans per kernel family), home solve in line, outside the timed region -- the timed region itself runs
    # from captured graphs, which cannot hold event nodes
    hbm_peak, peak_src = measured_peaks()
    bf16_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops_sustained", 1346.3) \
        if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 1400.0
    ev_frac = float(hm["has_ev"].mean())
    window = float(np.mean((hm["end"] - hm["start"])[hm["has_ev"] > 0])) / T if ev_frac > 0 else 0.0
    n_p = [(n + 15) // 16 * 16 for n in sizes]
    Hp = sum(n_p)
    # DESIGN.md kernel table: EV home reads load + (P_est,P_sch,Gamma inside the plug-in window), writes P_sch',P_ev
    home_bytes = Hp * T * (ev_frac * (8 + 24 * window + 16) + (1 - ev_frac) * 24)
    gemm_flops = sum(2.0 * n * n * T for n in n_p)
    f64_peak = fp64_gemm_peak_tflops() if rank == 0 else 0.0
    kernels = {}
    s1 = R.PipelinedSolver(sizes, T, device=local_rank, pipelines=1)
    s1.set_feeder_trees(trees)
    s1.set_homes(**hm_p)
    s1.set_tariff(cost_p)
    s1.set_option("overlap_home", 0)
    s1.set_option("graph", 0)
    s1.solve_admm(**ADMM)
    s1.solve_admm(**ADMM)
    st_iso = s1.stats()
    n_pipe = last.get("pipelines", 1)
    it = ADMM["iter_max"]
    iso_note = "extra single-pipeline solve, host-driven loop, home solve in line, outside the timed region (the timed region runs from captured graphs)"
    if st_iso["home_ms"] > 0:
        ms = st_iso["home_ms"] / it
        kernels["home_solve"] = {"bound": "hbm", "ms_per_launch": ms, "achieved": home_bytes / (ms * 1e-3) / 1e9,
                                 "peak": hbm_peak, "unit": "GB/s", "bytes_per_launch": home_bytes, "note": iso_note}
    if st_iso["dual_ms"] > 0:
        ms = st_iso["dual_ms"] / it
        # reads P_est (time-major), P_sch, Gamma; writes Gamma, P_est (home-major), z and g = [z]_+ with its bf16 copy for
        # the next utility solve (the previous schedule is not read: home_solve leaves the dual residual sums per home)
        dual_bytes_now = Hp * T * (24 + 24 + 8 + 2)
        kernels["dual_update"] = {"bound": "hbm", "ms_per_launch": ms, "achieved": dual_bytes_now / (ms * 1e-3) / 1e9,
                                  "peak": hbm_peak, "unit": "GB/s", "bytes_per_launch": dual_bytes_now, "note": iso_note}
    if st_iso["gemm_full_launches"] > 0 and st_iso["gemm_full_ms"] > 0:
        ms = st_iso["gemm_full_ms"] / st_iso["gemm_full_launches"]
        sbytes = sum(2.0 * n * n for n in n_p) + Hp * T * (2 + 4)
        kernels["screen_tc5"] = {"bound": "hbm", "ms_per_launch": ms, "achieved": sbytes / (ms * 1e-3) / 1e9,
                                 "peak": hbm_peak, "unit": "GB/s", "tflops": gemm_flops / (ms * 1e-3) / 1e12,
                                 "tensor_peak_tflops": bf16_peak, "bytes_per_launch": sbytes,
                                 "launches_per_step": st_iso["gemm_launches"], "ms_total_per_step": st_iso["gemm_ms"], "note": iso_note}
    roofline = None
    dom_name = "utility_qp_warp_kernel"
    n_mean = Hp / max(len(sizes), 1)
    if st_iso["qp_ms"] > 0:
        # Algorithmic HBM bytes (DESIGN.md section 3): a column that enters a QP kernel reads z, g, the screened voltages and
        # its multipliers and writes g, its bf16 copy and the multipliers back: 38 B per residence; every column costs its
        # work-list flags (16 B) per round.
        rest = st_iso["gemm_ms"] + st_iso["dual_ms"] + st_iso["home_ms"]
        qp_wall = max(st_iso["total_ms"] - rest, 1e-9)
        qp_bytes = st_iso["qp_columns"] * n_mean * 38.0 + st_iso["qp_outer_iterations"] * len(sizes) * T * 16.0
        kernels["utility_qp"] = {"bound": "hbm", "note": "active-set solver, latency-bound (one warp or one CTA per (zone,hour) column); " + iso_note,
                                 "ms_wall_per_step": qp_wall, "achieved": qp_bytes / (qp_wall * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "bytes_per_step": qp_bytes, "columns_solved_per_step": st_iso["qp_columns"],
                                 "fp64_tflops": st_iso["qp_flops"] / (qp_wall * 1e-3) / 1e12, "fp64_peak_tflops": f64_peak,
                                 "ms_warp_kernels": st_iso["qp_warp_ms"], "ms_init_kernel": st_iso["qp_init_ms"],
                                 "ms_cta_classes": st_iso["qp_ms"] - st_iso["qp_warp_ms"] - st_iso["qp_init_ms"]}
        if st_iso["qp_warp_rounds"] > 0 and st_iso["qp_warp_ms"] > 0:
            rounds_w = st_iso["qp_warp_rounds"]
            ms_round = st_iso["qp_warp_ms"] / rounds_w
            bytes_round = st_iso["qp_columns"] * n_mean * 38.0 / rounds_w
            traffic = None
            for name in ("traffic_r02.json", "traffic_r01.json"):     # dram bytes from the committed ncu --set full capture
                tp = os.path.join(ROOT, "profiles", name)
                if os.path.exists(tp):
                    try:
                        traffic = json.load(open(tp)).get("utility_qp_warp_kernel_bytes_per_round")
                    except Exception:
                        traffic = None
                    break
            ach = bytes_round / (ms_round * 1e-3) / 1e9
            roofline = {"kernel": dom_name, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                        "traffic": traffic, "ms_per_launch_group": ms_round, "bytes_per_launch_group": bytes_round,
                        "launch_groups_per_step": rounds_w, "peak_source": peak_src,
                        "note": "dominant kernels by time: the warp-per-column QP kernels (one launch per zone-size group and working-set "
                                "round, timed as a group with CUDA events on the utility stream).  An active-set solver, latency-bound by "
                                "construction (DESIGN.md section 3); the HBM-bound kernels of the path are in `kernels`"}
    # FP64 DMMA contraction (reliability check / exact mode): one extra solve outside the timed region
    if rank == 0 and not args.no_exact:
        s1.set_option("screen", 0)
        s1.set_option("overlap_home", 1)
        s1.solve_admm(**ADMM)
        st = s1.stats()
        if st["gemm_full_launches"] > 0:
            ms = st["gemm_full_ms"] / st["gemm_full_launches"]
            kernels["contract_f64"] = {"bound": "tensor", "ms_per_launch": ms, "achieved": gemm_flops / (ms * 1e-3) / 1e12,
                                       "peak": f64_peak, "unit": "TFLOP/s",
                                       "peak_source": "cuBLAS DGEMM 6144^3 measured in this run",
                                       "note": "exact mode (screen=0), single pipeline, measured outside the timed region",
                                       "ms_per_step_exact_mode": st["total_ms"]}
    s1.close()
    for k in kernels.values():
        if "peak" in k and k["peak"]:
            k["frac"] = k["achieved"] / k["peak"]
    tot = max(st_iso["total_ms"], 1e-9)
    share = {"screen_tc5": st_iso["gemm_ms"] / tot, "home_solve(in line)": st_iso["home_ms"] / tot, "dual_update": st_iso["dual_ms"] / tot,
             "utility_qp": max(0.0, 1.0 - (st_iso["gemm_ms"] + st_iso["dual_ms"] + st_iso["home_ms"]) / tot),
             "of": "device time of the host-driven single-pipeline solve (%.2f ms)" % st_iso["total_ms"]}

    cpu = None
    big_zone = workload_shape(args.workload)[1] > 4000
    if rank == 0 and world == 1 and not args.no_cpu_baseline and big_zone and args.cpu_sample_feeders is None:
        # one 10k-home zone: the dense CPU port needs a 0.8 GB matrix and minutes per ADMM iteration; timed only on request
        cpu = {"value": None, "unit": "home-hours/s", "cores": os.cpu_count() or 1, "kind": "port",
               "sample": "not timed by default for this workload (dense 10k x 10k port: minutes per ADMM iteration); pass --cpu-sample-feeders 1"}
    elif rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, dt, desc = cpu_port_sample(args.workload, args.cpu_sample_feeders, no_split=args.no_split)
        cpu = {"value": v, "unit": "home-hours/s", "cores": os.cpu_count() or 1, "kind": "port", "sample": desc,
               "seconds": dt}

    if rank == 0:
        nf, n, _ = workload_shape(args.workload)
        spread = [r[0] for r in per_rank]
        line = {
            "metric": "home_hours_scheduled_per_sec", "value": value, "unit": "home-hours/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload, "feeders_per_gpu": (nf // world if strong else nf), "feeders_total": nf if strong else nf * world,
                       "homes_per_feeder": n, "T": T, "pipelines_per_gpu": n_pipe,
                       "voltage_zones_rank0": len(sizes), "zone_sizes_rank0": [int(min(sizes)), int(max(sizes))], "homes_total": int(total_homes), **ADMM,
                       "population": ("one fixed population cut into %d contiguous shares" % world) if strong
                                     else "every rank draws its own population (seed = rank)",
                       "loop": "whole schedule from one captured CUDA graph per pipeline (device-side while loops)",
                       "l2": "working set per solve > L2 (sensitivity blocks %.2f GB on rank 0)" % (sum(8.0 * x * x for x in n_p) / 1e9)},
            "admm_iters_per_sec": ADMM["iter_max"] / (ms_step * 1e-3),
            "home_steps_per_sec": total_homes * T / (ms_step * 1e-3),
            "device_ms_per_step": dev_ms / args.steps,
            "per_rank_ms": {"columns": ["wall (CUDA events)", "host wall of solve_admm", "device span of the ADMM loop"], "rows": per_rank,
                            "max_over_min": max(spread) / max(min(spread), 1e-9)},
            "e2e": {"value": e2e_value, "unit": "home-hours/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "results": "P_sch + charging bit masks + diff (revs_get_schedule); P_ev / SOC rebuilt from the masks on request",
                    "compact_equals_full": compact_ok},
            "gpu_launches": int(stats_acc["kernel_launches"]),
            "roofline": roofline, "kernels": kernels, "share_of_device_time": share, "dominant_kernel": dom_name,
            "qp": {"outer_rounds_per_step": stats_acc["qp_outer_iterations"] / args.steps,
                   "newton_steps_per_step": stats_acc["qp_newton_iterations"] / args.steps,
                   "max_working_set": last["max_working_set"]},
            "residuals": {"primal": last["primal_residual"], "dual": last["dual_residual"]},
            "convergence": conv,
            "objective_check": {"distributed_cost": oc_dist, "cost_lower_bound_without_voltage_limits": oc_lb,
                                "rel_gap": (oc_dist - oc_lb) / max(abs(oc_lb), 1e-300),
                                "max_voltage_violation_of_P_sch_pu2_sampled_zones": oc_viol,
                                "upper_half_valid": bool(oc_viol <= 1e-9),
                                "note": "lower bound (cheapest SOC-feasible schedule of every home without voltage rows) <= optimum of the "
                                        "SOC-targeted centralized program <= distributed cost where P_sch is voltage-feasible.  The operator "
                                        "estimate P_est always satisfies the rows (tests); the homes' own schedule P_sch after iter_max "
                                        "iterations of the reference's algorithm need not (violation over the first 64 zones of every rank).  "
                                        "The reference's solve_central itself has no SOC target: lpsolver.solve_central reproduces its file"},
            "clocks": clk.summary(), "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    s.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="graft", choices=["graft", "reference"])
    ap.add_argument("--workload", default="synthetic-refshape-125k-homes-per-gpu-x96", choices=list(WORKLOADS))
    ap.add_argument("--cpu-sample-feeders", type=int, default=None, help="feeders of the workload the CPU port is timed on (default: 4 per core)")
    ap.add_argument("--pipelines", type=int, default=4, help="independent stream pipelines per GPU (parallel.PipelinedSolver)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-exact", action="store_true", help="skip the extra exact-mode (FP64 contraction) solve used for the contract_f64 figure")
    ap.add_argument("--no-split", action="store_true", help="hand whole feeders to the solver instead of their voltage zones")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="strong: the workload's feeders are one fixed population cut over the ranks")
    ap.add_argument("--tol", type=float, default=1e-3, help="stopping rule of the convergence leg (both ADMM residuals, kW)")
    ap.add_argument("--conv-iter-max", type=int, default=100)
    ap.add_argument("--no-convergence", action="store_true", help="skip the convergence leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed device-resident steps, write rank 0's results of the last step as DIR/<name>.npy "
                         "(float64; a fixed sample of %d homes of larger populations)" % DUMP_HOMES)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the GPU path (--impl graft)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()

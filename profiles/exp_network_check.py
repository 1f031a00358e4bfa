"""Cost of the population network check (revs_network_check) on the bench's default population, against the per-zone
revs_reliability loop it replaces, and the worst voltage-row excess of the whole population next to the 64-zone
sample of bench.py.  One GPU; writes one JSON (--out).

    python profiles/exp_network_check.py --out profiles/exp_network_check_b200.json

Times: `call_ms` is the host clock around the synchronous call (it ends in a stream synchronise; the full-array variant
includes the two device-to-host copies of [nodes, T] float64 into pageable memory); `kernel_ms` is the device time of
the check's kernels from a torch.profiler (CUPTI) pass of its own, summed per call.  The achieved bandwidth counts
the bytes the algorithm needs: the schedule read once, the outputs written once."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ADMM = dict(kappa=5.0, iter_max=15, vset=1.03, vlow=0.95, vhigh=1.05)   # bench.py
HBM_BYTES_PER_S = 7.7e12                                                 # HGX B200 data sheet, one GPU
KERNELS = ("network_check_kernel", "network_reduce_kernel")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power)


def stats_ms(xs):
    xs = np.asarray(xs)
    return dict(median=float(np.median(xs)), min=float(xs.min()), max=float(xs.max()), p10=float(np.percentile(xs, 10)),
                p90=float(np.percentile(xs, 90)), n=int(len(xs)))


def timed_calls(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append(1e3 * (time.perf_counter() - t0))
    return out


def kernel_ms(fn, reps):
    """Device time of the check's kernels per call (CUPTI activity records, a run of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    per = {k: [] for k in KERNELS}
    for ev in prof.events():
        for k in KERNELS:
            if k in ev.name and ev.device_type.name == "CUDA":
                per[k].append((ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3)
    return dict(mean_per_call_ms=sum(sum(v) for v in per.values()) / reps,
                per_launch_ms={k: stats_ms(v) for k, v in per.items() if v},
                launches_per_call={k: len(v) / reps for k, v in per.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "exp_network_check_b200.json"))
    ap.add_argument("--feeders", type=int, default=125)
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    import torch
    import revs_admm_b200 as R
    from revs_admm_b200.feeder import population
    torch.cuda.init()
    res = dict(gpu=gpu_info(), population=f"refshape x {args.feeders} feeders, T=96, seed 0", admm=ADMM)

    trees, hm, cost, sizes, T = population("refshape", args.feeders, seed=0)
    H, N = sum(sizes), sum(t.n_nodes for t in trees)
    res.update(zones=len(trees), homes=H, nodes=N, T=T)
    s = R.Solver(sizes, T)
    s.set_feeder_trees(trees)
    s.set_homes(**hm)
    s.set_tariff(cost)
    t0 = time.perf_counter()
    s.solve_admm(**ADMM)
    res["solve_admm_wall_ms"] = 1e3 * (time.perf_counter() - t0)
    res["solve_admm_device_ms"] = s.stats()["total_ms"]
    kw = dict(vset=ADMM["vset"], vlow=ADMM["vlow"], vhigh=ADMM["vhigh"])
    t0 = time.perf_counter()
    s.network_check("schedule", **kw)
    res["first_call_ms_incl_preparation"] = 1e3 * (time.perf_counter() - t0)

    summary_only = lambda: s.network_check("schedule", **kw)
    full = lambda: s.network_check("schedule", full=True, zones=True, **kw)
    res["summary_only"] = dict(call_ms=stats_ms(timed_calls(summary_only, args.reps)), kernel=kernel_ms(summary_only, args.reps))
    res["full_arrays"] = dict(call_ms=stats_ms(timed_calls(full, args.reps)), kernel=kernel_ms(full, args.reps))
    p_bytes, out_bytes = 8 * H * T, 2 * 8 * N * T
    for key, nbytes in (("summary_only", p_bytes), ("full_arrays", p_bytes + out_bytes)):
        ms = res[key]["kernel"]["mean_per_call_ms"]
        res[key]["algorithmic_bytes"] = nbytes
        res[key]["hbm_fraction_of_7.7TBps"] = nbytes / (ms * 1e-3) / HBM_BYTES_PER_S

    # the worst voltage row of the whole population vs bench.py's 64-zone host sample
    u = ADMM["vhigh"] ** 2 - ADMM["vset"] ** 2
    P_sch = s.results()["P_sch"]
    P_est = s.estimate()[0]
    off = np.concatenate([[0], np.cumsum(sizes)])
    sample = max(float((tr.drop(P_sch[off[z]:off[z + 1]]) - u).max()) for z, tr in enumerate(trees[:64]))
    res["row_excess"] = dict(P_sch=s.network_check("schedule", **kw)["summary"],
                             P_est=s.network_check("estimate", **kw)["summary"],
                             P_sch_bench_sample_64_zones_host=sample)

    # what the check replaces: revs_reliability zone by zone, voltage + flow of every node (run once)
    full_out = s.network_check("schedule", full=True, **kw)
    t0 = time.perf_counter()
    worst_dv = worst_df = 0.0
    a = 0
    for f, tr in enumerate(trees):
        rows = np.arange(tr.n_nodes)
        v = s.reliability(f, R.REVS_REL_VOLTAGE, rows, vset=ADMM["vset"])
        fl = s.reliability(f, R.REVS_REL_FLOW, rows)
        worst_dv = max(worst_dv, float(np.abs(v - full_out["voltage"][a:a + tr.n_nodes]).max()))
        worst_df = max(worst_df, float(np.abs(fl - full_out["loading"][a:a + tr.n_nodes]).max()))
        a += tr.n_nodes
    res["reliability_loop"] = dict(wall_ms_incl_comparison=1e3 * (time.perf_counter() - t0), calls=2 * len(trees),
                                   max_abs_diff_voltage=worst_dv, max_abs_diff_flow=worst_df)
    s.close()

    # config-3 zone: one 10,000-home radial feeder, 14,100 nodes (voltage only, once each)
    trees, hm, cost, sizes, T = population("radial10k", 1, seed=0)
    s = R.Solver(sizes, T)
    s.set_feeder_trees(trees)
    P = np.random.default_rng(0).uniform(0.0, 3.0, (sum(sizes), T))
    s.network_check(P, vset=ADMM["vset"])                 # breadth-first arrays built here
    t0 = time.perf_counter()
    v_net = s.network_check(P, vset=ADMM["vset"], full=True)["voltage"]
    t_net = 1e3 * (time.perf_counter() - t0)
    t0 = time.perf_counter()
    v_rel = s.reliability(0, R.REVS_REL_VOLTAGE, np.arange(trees[0].n_nodes), vset=ADMM["vset"], P=P)
    t_rel = 1e3 * (time.perf_counter() - t0)
    res["config3_zone"] = dict(nodes=trees[0].n_nodes, homes=sum(sizes), network_check_full_call_ms=t_net,
                               reliability_voltage_call_ms=t_rel, max_abs_diff_voltage=float(np.abs(v_net - v_rel).max()),
                               kernel=kernel_ms(lambda: s.network_check(P, vset=ADMM["vset"]), 20))
    s.close()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1, default=float)
    print(json.dumps(res, indent=1, default=float))


if __name__ == "__main__":
    main()

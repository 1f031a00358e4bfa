"""The greedy voltage repair (revs_repair_schedule) on the bench's default population after the bench's 15-iteration
solve_admm: its time, the zones it repairs and leaves, its moves and drops, the tariff cost of the repaired schedule
against bench.objective_check's lower bound, and the repaired schedule's network summary.  Also the config-3
radial10k zone, once.  One GPU; writes one JSON (--out).

    python profiles/exp_repair.py --out profiles/exp_repair_b200.json

Times: `call_ms` is the host clock around the synchronous call (summary outputs only: zone_info); `kernel` is the device
time of the call's kernels (the network check that gives the initial drops, and the repair) from a torch.profiler
(CUPTI) pass of its own, summed per call, after warm-up calls."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from exp_network_check import ADMM, gpu_info, stats_ms, timed_calls  # noqa: E402

KERNELS = ("network_check_kernel", "network_reduce_kernel", "repair_kernel")


def kernel_ms(fn, reps):
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


def brief(r):
    return {k: r[k] for k in ("moves", "drops", "zones_violated", "zones_repaired", "zones_left")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "exp_repair_b200.json"))
    ap.add_argument("--feeders", type=int, default=125)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import torch
    import bench
    import revs_admm_b200 as R
    from revs_admm_b200.feeder import population
    torch.cuda.init()
    res = dict(gpu=gpu_info(), population=f"refshape x {args.feeders} feeders, T=96, seed 0", admm=ADMM)
    kw = dict(vset=ADMM["vset"], vhigh=ADMM["vhigh"])

    trees, hm, cost, sizes, T = population("refshape", args.feeders, seed=0)
    res.update(zones=len(trees), homes=sum(sizes), T=T)
    s = R.Solver(sizes, T)
    s.set_feeder_trees(trees)
    s.set_homes(**hm)
    s.set_tariff(cost)
    s.solve_admm(**ADMM)
    t0 = time.perf_counter()
    rep = s.repair_schedule(mask=True, **kw)
    res["first_call_ms_incl_preparation"] = 1e3 * (time.perf_counter() - t0)
    res["repair"] = brief(rep)
    info_only = lambda: s.repair_schedule(schedule=False, **kw)
    res["call_ms"] = stats_ms(timed_calls(info_only, args.reps))
    res["kernel"] = kernel_ms(info_only, args.reps)
    net = dict(vset=ADMM["vset"], vlow=ADMM["vlow"], vhigh=ADMM["vhigh"])
    res["network_summary"] = dict(schedule=s.network_check("schedule", **net)["summary"],
                                  repaired=s.network_check("repaired", **net)["summary"])
    P_sch = s.results(want_diff=False)["P_sch"]
    dist_cost, lb, _ = bench.objective_check(trees, hm, cost, P_sch, T)
    rep_cost = float((rep["P_sch"] @ cost).sum())
    res["tariff_cost"] = dict(P_sch=dist_cost, repaired=rep_cost, lower_bound_without_voltage_limits=lb,
                              repaired_gap_to_lower_bound=(rep_cost - lb) / lb,
                              repaired_is_valid_upper_bound=rep["zones_left"] == 0)
    s.close()

    # config-3 zone: one 10,000-home radial feeder (global-memory state), once
    trees, hm, cost, sizes, T = population("radial10k", 1, seed=0)
    s = R.Solver(sizes, T)
    s.set_feeder_trees(trees)
    s.set_homes(**hm)
    s.set_tariff(cost)
    s.solve_admm(**ADMM)
    s.network_check("schedule", **net)                       # breadth-first arrays built here
    t0 = time.perf_counter()
    rep = s.repair_schedule(schedule=False, **kw)
    res["config3_zone"] = dict(homes=sum(sizes), call_ms=1e3 * (time.perf_counter() - t0), repair=brief(rep),
                               network_summary_repaired=s.network_check("repaired", **net)["summary"])
    s.close()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1, default=float)
    print(json.dumps(res, indent=1, default=float))


if __name__ == "__main__":
    main()

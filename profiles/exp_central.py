"""The bracket of the centralized optimum (revs_central_bracket) on the bench's default population, after the bench's
15-iteration solve_admm: device time per call split into the repairs and the rest (ascent, selections, network
checks), zones per status, sum LB and sum UB against bench.objective_check's bound, the cost of P_sch and of the
repaired ADMM schedule, and the gap for several ascent lengths.  One GPU; writes one JSON (--out).

    python profiles/exp_central.py --out profiles/exp_central_b200.json

Times: `call_ms` is the host clock around the synchronous call (summary outputs only: zone_bounds, zone_info);
`kernel` is the device time of the call's kernels from a torch.profiler (CUPTI) pass of its own, after a warm-up call."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from exp_network_check import ADMM, gpu_info, stats_ms, timed_calls  # noqa: E402

REPAIR = ("repair_kernel",)
ASCENT = ("network_check_kernel", "network_reduce_kernel", "central_select_kernel", "central_ascent_kernel",
          "central_cost_kernel", "central_final_kernel")


def kernel_ms(fn, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    rep = asc = 0.0
    launches = 0
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        ms = (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
        if any(k in ev.name for k in REPAIR):
            rep += ms
            launches += 1
        elif any(k in ev.name for k in ASCENT):
            asc += ms
            launches += 1
    return dict(per_call_ms=(rep + asc) / reps, repairs_ms=rep / reps, ascent_and_rest_ms=asc / reps,
                launches_per_call=launches / reps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "exp_central_b200.json"))
    ap.add_argument("--feeders", type=int, default=125)
    ap.add_argument("--iters", default="0,50,100,200")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import numpy as np
    import torch
    import bench
    import revs_admm_b200 as R
    from revs_admm_b200.feeder import population
    torch.cuda.init()
    res = dict(gpu=gpu_info(), population=f"refshape x {args.feeders} feeders, T=96, seed 0", admm=ADMM)
    kw = dict(vset=ADMM["vset"], vhigh=ADMM["vhigh"])
    net = dict(vset=ADMM["vset"], vlow=ADMM["vlow"], vhigh=ADMM["vhigh"])

    trees, hm, cost, sizes, T = population("refshape", args.feeders, seed=0)
    res.update(zones=len(trees), homes=sum(sizes), T=T)
    s = R.Solver(sizes, T)
    s.set_feeder_trees(trees)
    s.set_homes(**hm)
    s.set_tariff(cost)
    s.solve_admm(**ADMM)
    P_sch = s.results(want_diff=False)["P_sch"]
    rep = s.repair_schedule(**kw)
    dist_cost, lb0, _ = bench.objective_check(trees, hm, cost, P_sch, T)
    res["reference_costs"] = dict(objective_check_lower_bound=lb0, P_sch=dist_cost,
                                  repaired_admm=float((rep["P_sch"] @ cost).sum()),
                                  repaired_admm_zones_left=rep["zones_left"])
    runs = {}
    for it in [int(x) for x in args.iters.split(",")]:
        t0 = time.perf_counter()
        r = s.central_bracket(iters=it, **kw)
        first_ms = 1e3 * (time.perf_counter() - t0)
        chk = s.network_check("central", zones=True, **net)
        st = r["zone_info"][:, 0]
        info_only = lambda: s.central_bracket(iters=it, schedule=False, **kw)    # noqa: E731
        runs[it] = dict(zones_status=r["zones_status"], lb_all_zones=r["lb"], lb_bracketed=r["lb_bracketed"],
                        ub_bracketed=r["ub"], gap_bracketed=r["gap"],
                        ub_cost_of_kept_schedule=float((r["P_sch"] @ cost).sum()),
                        lb_over_objective_check=(r["lb"] - lb0) / lb0,
                        ascent_steps=int(r["zone_info"][:, 1].sum()), repair_moves_drops=int(r["zone_info"][:, 2].sum()),
                        violated_rows_in_bracketed_zones=int((chk["zone_worst"][st <= 1, 1] > 1e-9).sum()),
                        first_call_ms=first_ms, call_ms=stats_ms(timed_calls(info_only, args.reps, warmup=1)),
                        kernel=kernel_ms(info_only, args.reps))
        print(it, json.dumps(runs[it], default=float), flush=True)
    res["central_bracket"] = runs
    after = s.results(want_diff=False)["P_sch"]
    res["admm_schedule_unchanged"] = bool(np.array_equal(after, P_sch))
    s.close()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1, default=float)
    print(json.dumps(res, indent=1, default=float))


if __name__ == "__main__":
    main()

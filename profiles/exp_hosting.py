"""The hosting capacity (revs_hosting_capacity) on the bench's default population after one ADMM run, and on the
radial10k zone: device time per call for counts only, with zone_uniform, with the [H, T] download of home_cap and with
a seeded line rating on every edge, next to the network check of the same schedule; and the share of plug-in window
steps where one more charger fits, for P_sch, the repaired schedule and the central bracket's schedule.  One GPU;
writes one JSON (--out).

    python profiles/exp_hosting.py --out profiles/exp_hosting_b200.json

Times: `call_ms` is the host clock around the synchronous call (the home_cap variant includes the device-to-host copy
of [H, T] float64 into pageable memory); `kernel` is the device time of the call's kernels from a torch.profiler
(CUPTI) pass of its own over `reps` calls after a warm-up call, per call and per kernel.  The seeded ratings are
1 / uniform(20, 400) kW per edge (seed 0), signs random: the population has no line data of its own."""
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

HOSTING = ("hosting_kernel", "hosting_reduce_kernel", "pack_rows_kernel")
NETWORK = ("network_check_kernel", "network_reduce_kernel")


def kernel_ms(fn, reps, names):
    """Device time of the call's kernels (CUPTI activity records), per call and per kernel name."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    per = {k: [] for k in names}
    for ev in prof.events():
        for k in names:
            if ev.device_type.name == "CUDA" and k in ev.name:
                per[k].append((ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3)
    return dict(mean_per_call_ms=sum(sum(v) for v in per.values()) / reps,
                per_kernel_ms={k: stats_ms(v) for k, v in per.items() if v},
                launches_per_call={k: len(v) / reps for k, v in per.items() if v})


def _shares(r):
    return dict(window_steps=r["window_steps"], window_steps_open=r["window_steps_open"],
                open_share=r["window_steps_open"] / max(r["window_steps"], 1), thermal_bound=r["thermal_bound"],
                home_cap_min=r["home_cap_min"], uniform_min=r["uniform_min"])


def one_population(name, feeders, reps, tools):
    import revs_admm_b200 as R
    from revs_admm_b200.feeder import population
    lim = dict(vset=ADMM["vset"], vhigh=ADMM["vhigh"])
    trees, hm, cost, sizes, T = population(name, feeders, seed=0)
    N = sum(t.n_nodes for t in trees)
    rng = np.random.default_rng(0)
    scale = rng.choice([-1.0, 1.0], N) / rng.uniform(20.0, 400.0, N)
    out = dict(population=f"{name} x {feeders} feeders, T={T}, seed 0", zones=len(trees), homes=sum(sizes),
               nodes=N, largest_zone=max(sizes), limits=lim, row_tol=1e-9)
    s = R.Solver(sizes, T)
    s.set_feeder_trees(trees)
    s.set_homes(**hm)
    s.set_tariff(cost)
    s.solve_admm(**ADMM)
    t0 = time.perf_counter()
    first = s.hosting_capacity("schedule", homes=False, **lim)
    out["first_call_ms"] = 1e3 * (time.perf_counter() - t0)
    variants = dict(counts_only=dict(homes=False, uniform=False), uniform=dict(homes=False, uniform=True),
                    home_cap_download=dict(homes=True, uniform=True),
                    seeded_scale=dict(homes=False, uniform=True, scale=scale))
    out["variants"] = {}
    for vname, kw in variants.items():
        fn = lambda: s.hosting_capacity("schedule", **kw, **lim)    # noqa: E731
        out["variants"][vname] = dict(call_ms=stats_ms(timed_calls(fn, reps, warmup=1)),
                                      kernel=kernel_ms(fn, reps, HOSTING))
    fn = lambda: s.network_check("schedule", vlow=ADMM["vlow"], **lim)     # noqa: E731
    out["network_check"] = dict(call_ms=stats_ms(timed_calls(fn, reps, warmup=1)), kernel=kernel_ms(fn, reps, NETWORK))
    a = s.hosting_capacity("schedule", scale=scale, **lim)
    b = s.hosting_capacity("schedule", scale=scale, **lim)
    out["two_calls_same_bytes"] = all(a[k].tobytes() == b[k].tobytes()
                                      for k in ("home_cap", "zone_uniform", "zone_counts"))
    out["counts_only_equal_full"] = bool(first["zone_counts"].tobytes() ==
                                         s.hosting_capacity("schedule", **lim)["zone_counts"].tobytes())
    if tools:
        s.repair_schedule(schedule=False, **lim)
        s.central_bracket(iters=100, schedule=False, **lim)
        out["schedules"] = {src: dict(no_scale=_shares(s.hosting_capacity(src, homes=False, **lim)),
                                      seeded_scale=_shares(s.hosting_capacity(src, homes=False, scale=scale, **lim)))
                            for src in ("schedule", "repaired", "central")}
    s.close()
    print(name, json.dumps(out, default=float), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "exp_hosting_b200.json"))
    ap.add_argument("--feeders", type=int, default=125)
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    res = dict(gpu=gpu_info())
    res["default"] = one_population("refshape", args.feeders, args.reps, True)
    res["radial10k"] = one_population("radial10k", 1, args.reps, False)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1, default=float)
    print(json.dumps(res, indent=1, default=float))


if __name__ == "__main__":
    main()

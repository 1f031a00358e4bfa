"""The certificate of voltage infeasibility (revs_certify_infeasible) on the bench's default population and on the
radial10k zone: device time per call, zones per kind, and, joined with central_bracket(iters=100), the bracket's status
table before and after central_status (how many of the zones the bracket leaves open get a certificate).  One GPU;
writes one JSON (--out).

    python profiles/exp_certify.py --out profiles/exp_certify_b200.json

Times: `call_ms` is the host clock around the synchronous call, after a warm-up call; `kernel` is the device time of the
call's kernels from a torch.profiler (CUPTI) pass of its own, one value per call, after a warm-up call."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from exp_network_check import ADMM, gpu_info, stats_ms, timed_calls  # noqa: E402

KERNELS = ("network_check_kernel", "network_reduce_kernel", "certify_base_kernel", "certify_count_kernel",
           "certify_final_kernel")


def kernel_ms(fn, reps):
    """Device time of the call's kernels, per call and per kernel name (CUPTI activity records)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    per_call = []
    by_name = {}
    for _ in range(reps):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        tot = 0.0
        for ev in prof.events():
            if ev.device_type.name != "CUDA" or not any(k in ev.name for k in KERNELS):
                continue
            ms = (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
            tot += ms
            name = next(k for k in KERNELS if k in ev.name)
            by_name[name] = by_name.get(name, 0.0) + ms / reps
        per_call.append(tot)
    return dict(per_call_ms=stats_ms(per_call), by_kernel_ms=by_name)


def one_population(name, feeders, reps, bracket_iters):
    import numpy as np
    import revs_admm_b200 as R
    from revs_admm_b200.feeder import population
    kw = dict(vset=ADMM["vset"], vhigh=ADMM["vhigh"])
    trees, hm, cost, sizes, T = population(name, feeders, seed=0)
    out = dict(population=f"{name} x {feeders} feeders, T={T}, seed 0", zones=len(trees), homes=sum(sizes),
               largest_zone=max(sizes), limits=kw, row_tol=1e-9)
    s = R.Solver(sizes, T)
    s.set_feeder_trees(trees)
    s.set_homes(**hm)
    s.set_tariff(cost)
    t0 = time.perf_counter()
    c = s.certify_infeasible(**kw)
    out["first_call_ms"] = 1e3 * (time.perf_counter() - t0)
    fn = lambda: s.certify_infeasible(**kw)    # noqa: E731
    out["call_ms"] = stats_ms(timed_calls(fn, reps, warmup=1))
    out["kernel"] = kernel_ms(fn, reps)
    again = s.certify_infeasible(**kw)["zone_cert"]
    out["two_calls_same_bytes"] = bool(again.tobytes() == c["zone_cert"].tobytes())
    kind = c["zone_cert"][:, 0]
    out["zones_kind"] = c["zones_kind"]
    out["certified"] = c["certified"]
    k2 = c["zone_cert"][kind == 2]
    out["kind2_k_histogram"] = {int(k): int((k2[:, 2] == k).sum()) for k in np.unique(k2[:, 2])}
    out["kind2_deficit_max"] = int(k2[:, 3].max()) if len(k2) else 0
    if bracket_iters is not None:
        t0 = time.perf_counter()
        br = s.central_bracket(iters=bracket_iters, schedule=False, **kw)
        bracket_ms = 1e3 * (time.perf_counter() - t0)
        st0 = br["zone_info"][:, 0]
        st1 = R.central_status(br["zone_info"], c["zone_cert"])
        out["central_bracket"] = dict(
            iters=bracket_iters, host_ms=bracket_ms,
            status_before=[int((st0 == k).sum()) for k in range(4)],
            status_after=[int((st1 == k).sum()) for k in range(4)],
            open_zones_certified=int(((st0 == 2) & (kind > 0)).sum()),
            open_zones_certified_by_kind=[int(((st0 == 2) & (kind == k)).sum()) for k in (1, 2)],
            lagrangian_certified_also_counted=int(((st0 == 3) & (kind > 0)).sum()),
            lagrangian_certified_not_counted=int(((st0 == 3) & (kind == 0)).sum()),
            open_zones_left=[int(z) for z in np.nonzero(st1 == 2)[0]])
    s.close()
    print(name, json.dumps(out, default=float), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "exp_certify_b200.json"))
    ap.add_argument("--feeders", type=int, default=125)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--bracket-iters", type=int, default=100)
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    res = dict(gpu=gpu_info())
    res["default"] = one_population("refshape", args.feeders, args.reps, args.bracket_iters)
    res["radial10k"] = one_population("radial10k", 1, max(2, args.reps // 5), None)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1, default=float)
    print(json.dumps(res, indent=1, default=float))


if __name__ == "__main__":
    main()

"""One EnergyVirtualObservablesEnsemble.update on the 64 x 64 fine mesh of BASELINE config 2 (setup_physics(4, 4, 4, "ND"),
d = 4095 free dofs), N = 128 data points, RBF subspaces of m weighting functions, n_it Newton iterations per update:
the batched route (one rho launch + one gpde_vo_energy_step_f64 launch per iteration) against the member loop
(EnergyVirtualObservable.update per data point), in the same process, alternated after warm-up, on the same draws.

    python profiles/tools/time_energy_vo.py --out DIR [--reps R] [--warmup W]

Per case: CUDA-event and host-clock (around a device synchronise) time per update for both routes (median and min over
R updates), kernels and copies per update with their summed device time and that of the energy-step kernel alone
(torch.profiler, one profiled update per route, separate from the timed ones),
and the largest relative difference of the posterior means between the routes after all updates.  Prints one line per
case and writes DIR/time_energy_vo.json with the card name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import gpde_b200  # noqa: E402,F401
from gpde_b200 import VirtualObservables as VO  # noqa: E402
from gpde_b200.physics import BoundaryConditionEnsemble, setup_physics  # noqa: E402
from gpde_b200 import fem  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def build(ph, X_DG, bce, m, n_it, dev, batched):
    fom = ph['fom']
    qpe = VO.QuerryPointEnsemble.FromArrays(X_DG, bce, fom, device=dev)
    ens = VO.EnergyVirtualObservablesEnsemble(qpe, n_it, VO.RadialBasisFunctionSampler(qpe[0], 0.1, m), torch.double, dev)
    ens.force_temperature(0.5)
    ens.batched_update = batched
    return ens


def timed_update(ens, G, P, it):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    ens.update(G, P, it)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3


def count_launches(ens, G, P, it):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        ens.update(G, P, it)
        torch.cuda.synchronize()
    dev_events = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    copies = sum(1 for e in dev_events if e.name.startswith(("Memcpy", "Memset")))
    us = lambda evs: float(sum(e.time_range.elapsed_us() for e in evs))
    return {"kernels": len(dev_events) - copies, "copies": copies, "device_busy_us": us(dev_events),
            "energy_step_kernel_us": us([e for e in dev_events if "vo_energy_step_kernel" in e.name])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for time_energy_vo.json")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--N", type=int, default=128)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    ph = setup_physics(4, 4, 4, "ND")
    fom = ph['fom']
    N, d = args.N, fom.dim_out
    rng = np.random.RandomState(0)
    img = fem.sample_log_field(64, 64, 0.0, 1.0, 0.1, N, rng)
    X_DG = img.reshape(N, -1)[:, fom.mesh.pixel_of_cell()]
    bce = BoundaryConditionEnsemble(ph, N, "ND")
    G = torch.tensor(rng.normal(size=(N, d)), device=dev)
    P = torch.tensor(rng.uniform(1.0, 30.0, size=(N, d)), device=dev)
    result = {"gpu": gpu_info(), "mesh": "64x64 fine (setup_physics(4, 4, 4, 'ND'))", "d": d, "N": N,
              "reps": args.reps, "warmup": args.warmup, "cases": []}
    for m in (8, 32):
        for n_it in (1, 4):
            routes = {"batched": build(ph, X_DG, bce, m, n_it, dev, True), "members": build(ph, X_DG, bce, m, n_it, dev, False)}
            times = {k: [] for k in routes}
            for rep in range(args.warmup + args.reps):
                for name, ens in routes.items():           # alternated, each on the same draws
                    np.random.seed(1000 + rep)
                    ev, host = timed_update(ens, G, P, rep)
                    assert ens.last_update_route == name
                    if rep >= args.warmup:
                        times[name].append((ev, host))
            mb, mm = routes["batched"].mean, routes["members"].mean
            diff = float(((mb - mm).abs().max() / mm.abs().max()).item())
            launches = {}
            for name, ens in routes.items():
                np.random.seed(99)
                launches[name] = count_launches(ens, G, P, 0)
            case = {"m": m, "n_it": n_it, "max_rel_diff_mean": diff, "launches_per_update": launches}
            for name, tt in times.items():
                ev, host = np.array(tt).T
                case[name] = {"event_ms_median": float(np.median(ev)), "event_ms_min": float(ev.min()),
                              "host_ms_median": float(np.median(host)), "host_ms_min": float(host.min())}
            case["speedup_event_median"] = case["members"]["event_ms_median"] / case["batched"]["event_ms_median"]
            result["cases"].append(case)
            print("m=%2d n_it=%d  batched %.3f ms (host %.3f; device busy %.0f us, energy steps %.0f us)  members %.3f ms "
                  "(host %.3f)  x%.1f  kernels %d vs %d  max rel diff %.1e"
                  % (m, n_it, case["batched"]["event_ms_median"], case["batched"]["host_ms_median"],
                     launches["batched"]["device_busy_us"], launches["batched"]["energy_step_kernel_us"],
                     case["members"]["event_ms_median"], case["members"]["host_ms_median"], case["speedup_event_median"],
                     launches["batched"]["kernels"], launches["members"]["kernels"], diff), flush=True)
            del routes
    print("%s, power limit %s" % (result["gpu"]["name"], result["gpu"]["power_limit"]))
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "time_energy_vo.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()

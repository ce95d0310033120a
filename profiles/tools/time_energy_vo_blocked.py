"""One EnergyVirtualObservablesEnsemble.update with 64 < m <= 256 weighting functions per data point: the blocked route
(per Newton iteration one rho launch + gpde_vo_energy_step_blocked_f64, i.e. vo_energy_gram_kernel, vo_post_factor_kernel
and vo_energy_apply_kernel) against the member loop (EnergyVirtualObservable.update per data point), in the same process,
alternated after warm-up, on the same draws.

    python profiles/tools/time_energy_vo_blocked.py --out DIR [--reps R] [--warmup W]

Cases: the 64 x 64 fine mesh (setup_physics(4, 4, 4, "ND"), d = 4095) with N = 128, m in {96, 256}, n_it in {1, 4}, RBF
columns (l = 0.1) and Gaussian-sketch columns; the 128 x 128 fine mesh of config 3 (setup_physics(8, 8, 4, "ND"),
d = 16383) with m = 256, N = 32, n_it = 1, RBF columns.  Per case: the median and min of R CUDA-event timed updates per
route; from one separate torch.profiler update per route, the kernels per update and, on the blocked route, the device
time of each of its three kernels; the largest relative difference of the means after all updates.  An update that
raises (an M_n whose Cholesky meets a non-positive pivot on the blocked route) is recorded as such.  Prints one line per
case and writes DIR/r3_energy_vo_blocked_f64.json with the card name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import gpde_b200  # noqa: E402,F401
from gpde_b200 import VirtualObservables as VO  # noqa: E402
from gpde_b200.physics import BoundaryConditionEnsemble, setup_physics  # noqa: E402
from gpde_b200 import fem  # noqa: E402

KERNELS = ("vo_energy_gram_kernel", "vo_post_factor_kernel", "vo_energy_apply_kernel")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def build(ph, X_DG, bce, sampler, m, n_it, dev, route):
    qpe = VO.QuerryPointEnsemble.FromArrays(X_DG, bce, ph['fom'], device=dev)
    s = VO.RadialBasisFunctionSampler(qpe[0], 0.1, m) if sampler == "rbf" else VO.GaussianSketchingSampler(qpe[0], m)
    ens = VO.EnergyVirtualObservablesEnsemble(qpe, n_it, s, torch.double, dev)
    ens.force_temperature(0.5)
    ens.max_blocked_m = 256
    ens.batched_update = route == "blocked"
    return ens


def timed_update(ens, G, P, it):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    ens.update(G, P, it)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def profiled_update(ens, G, P, it):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ens.update(G, P, it)
        torch.cuda.synchronize()
    evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    copies = sum(1 for e in evs if e.name.startswith(("Memcpy", "Memset")))
    out = {"kernels": len(evs) - copies, "copies": copies,
           "device_busy_us": float(sum(e.time_range.elapsed_us() for e in evs))}
    for k in KERNELS:
        sel = [e.time_range.elapsed_us() for e in evs if k in e.name]
        if sel:
            out[k] = {"launches": len(sel), "us_total": float(sum(sel))}
    return out


def run_case(ph, N, sampler, m, n_it, reps, warmup, dev, rng):
    fom = ph['fom']
    d, nx = fom.dim_out, int(round(np.sqrt(fom.dim_in // 2)))
    img = fem.sample_log_field(nx, nx, 0.0, 1.0, 0.1, N, rng)
    X_DG = img.reshape(N, -1)[:, fom.mesh.pixel_of_cell()]
    bce = BoundaryConditionEnsemble(ph, N, "ND")
    G = torch.tensor(rng.normal(size=(N, d)), device=dev)
    P = torch.tensor(rng.uniform(1.0, 30.0, size=(N, d)), device=dev)
    routes = {r: build(ph, X_DG, bce, sampler, m, n_it, dev, r) for r in ("blocked", "members")}
    times = {r: [] for r in routes}
    case = {"mesh": "%dx%d" % (nx, nx), "d": d, "N": N, "sampler": sampler, "m": m, "n_it": n_it}
    try:
        for rep in range(warmup + reps):
            for name, ens in routes.items():              # alternated, each on the same draws
                np.random.seed(1000 + rep)
                ms = timed_update(ens, G, P, rep)
                assert ens.last_update_route == name
                if rep >= warmup:
                    times[name].append(ms)
    except RuntimeError as e:
        case["error"] = "%s update raised: %s" % (name, e)
        print("%s m=%d n_it=%d %s: %s" % (case["mesh"], m, n_it, sampler, case["error"]), flush=True)
        return case
    mb, mm = routes["blocked"].mean, routes["members"].mean
    case["max_rel_diff_mean"] = float(((mb - mm).abs().max() / mm.abs().max()).item())
    for name, tt in times.items():
        case[name] = {"event_ms_median": float(np.median(tt)), "event_ms_min": float(np.min(tt)), "event_ms": tt}
    case["speedup_event_median"] = case["members"]["event_ms_median"] / case["blocked"]["event_ms_median"]
    case["profile"] = {}
    for name, ens in routes.items():
        np.random.seed(99)
        case["profile"][name] = profiled_update(ens, G, P, 0)
    pb = case["profile"]["blocked"]
    print("%s m=%3d n_it=%d %-8s blocked %8.3f ms  members %9.3f ms  x%6.1f  kernels %d vs %d  gram %.0f us  factor %.0f us"
          "  apply %.0f us  max rel diff %.1e"
          % (case["mesh"], m, n_it, sampler, case["blocked"]["event_ms_median"], case["members"]["event_ms_median"],
             case["speedup_event_median"], pb["kernels"], case["profile"]["members"]["kernels"],
             pb[KERNELS[0]]["us_total"], pb[KERNELS[1]]["us_total"], pb[KERNELS[2]]["us_total"],
             case["max_rel_diff_mean"]), flush=True)
    return case


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for r3_energy_vo_blocked_f64.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    result = {"gpu": gpu_info(), "reps": args.reps, "warmup": args.warmup, "temperature": 0.5, "cases": []}
    rng = np.random.RandomState(0)
    ph = setup_physics(4, 4, 4, "ND")
    for sampler in ("rbf", "gauss"):
        for m in (96, 256):
            for n_it in (1, 4):
                result["cases"].append(run_case(ph, 128, sampler, m, n_it, args.reps, args.warmup, dev, rng))
    result["cases"].append(run_case(setup_physics(8, 8, 4, "ND"), 32, "rbf", 256, 1, args.reps, args.warmup, dev, rng))
    print("%s, power limit %s" % (result["gpu"]["name"], result["gpu"]["power_limit"]))
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r3_energy_vo_blocked_f64.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()

"""VirtualObservablesEnsemble.update (the precision hyper-update included) with 64 < m <= 256 weighting functions per data
point: the blocked route (gpde_vo_posterior_blocked_f64 + the panel moments kernel) against the dense route
(condition_gaussian on the materialised Gamma_n, forced with ``max_blocked_m = 64`` on the same ensemble instance).

    python profiles/tools/time_vo_posterior_blocked.py --out DIR [--reps R] [--warmup W] [--cases 128:256:32,...]

Cases (fine mesh : m : N), V = W of the coarse-grained-residual sampler + RBF columns (l = 0.1), one V per data point:
128 x 128 (setup_physics(8, 8, 4, "ND"), W = 81 columns) with m = 256 and N in {32, 128}; 64 x 64 (setup_physics(4, 4,
4, "ND"), W = 25 columns) with m in {96, 256} and N = 128.  Per case: CUDA-event time per update for both routes (median
and min of R alternated updates after W warm-ups; the dense route's first update, which materialises Gamma_n, is timed
on its own), per-kernel device time from a separate torch.profiler update per route, the achieved FP64 rate of the two
row passes of the blocked route (algorithmic work 2 nbt 64^2 d N per pass, nbt = lower 64 x 64 blocks), peak device
memory of one update per route, and the largest relative difference of mean and vars between the routes on the same
state.  Writes DIR/r3_vo_posterior_blocked.json with the card name and power limit."""
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

DMMA_PEAK_TFLOPS = 37.0      # measured FP64 DMMA rate of the card (profiles/r1_fp64_peak.txt)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def build(nx_rom, m, N, dev, seed=0):
    ph = setup_physics(nx_rom, nx_rom, 4, "ND")
    fom = ph['fom']
    rng = np.random.RandomState(seed)
    nf = fom.mesh.nx
    img = fem.sample_log_field(nf, nf, 0.0, 1.0, 0.1, N, rng)
    X_DG = img.reshape(N, -1)[:, fom.mesh.pixel_of_cell()]
    bce = BoundaryConditionEnsemble(ph, N, "ND", rng=rng)
    qpe = VO.QuerryPointEnsemble.FromArrays(X_DG, bce, fom, device=dev)
    n_w = ph['W'].shape[1]
    np.random.seed(seed)
    qe = VO.QuerryEnsemble.FromQuerryPointEnsemble(qpe, ph, CGR=True, flux=False, N_gaussian=0, N_rbf=m - n_w, l_rbf=0.1,
                                                   dtype=torch.double, device=dev)
    for q in qe:     # learnable precisions: the hyper-update runs its moments pass
        q._sampler.__class__ = type("Learnable", (q._sampler.__class__,), {"precision_mask": property(lambda s: np.ones(s.m))})
    ens = VO.VirtualObservablesEnsemble(qpe, qe, torch.double, dev)
    G = torch.tensor(rng.normal(size=(N, fom.dim_out)), device=dev)
    P = torch.tensor(rng.uniform(1.0, 30.0, size=(N, fom.dim_out)), device=dev)
    return ens, G, P, fom.dim_out


def set_route(ens, route):
    if route == "dense":
        ens.max_blocked_m = 64
    elif "max_blocked_m" in ens.__dict__:
        del ens.max_blocked_m


def timed_update(ens, G, P, it):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    ens.update(G, P, it)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def peak_update(ens, G, P, it):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    ms = timed_update(ens, G, P, it)
    return ms, torch.cuda.max_memory_allocated() - base, torch.cuda.memory_allocated() - base


def kernel_times(ens, G, P, it):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ens.update(G, P, it)
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            name = e.name if len(e.name) < 90 else e.name[:90]
            c = per.setdefault(name, [0, 0.0])
            c[0] += 1
            c[1] += e.time_range.elapsed_us()
    return {k: {"count": c, "us": round(t, 1)} for k, (c, t) in sorted(per.items(), key=lambda kv: -kv[1][1])}


def kernel_us(kt, key):
    return sum(v["us"] for k, v in kt.items() if key in k)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--cases", default="128:256:32,128:256:128,64:96:128,64:256:128")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    result = {"gpu": gpu_info(), "reps": args.reps, "warmup": args.warmup, "dmma_peak_tflops": DMMA_PEAK_TFLOPS,
              "cases": []}
    for spec in args.cases.split(","):
        nf, m, N = (int(v) for v in spec.split(":"))
        ens, G, P, d = build(8 if nf == 128 else 4, m, N, dev)
        assert ens.m == m
        it = 0
        for _ in range(1 + args.warmup):           # the first update initialises the precision hyper-update
            set_route(ens, "blocked"); timed_update(ens, G, P, it); it += 1
        assert ens.last_update_route == "blocked"
        _, peak_b, _ = peak_update(ens, G, P, it); it += 1
        set_route(ens, "dense")
        first_dense, peak_d, resident_d = peak_update(ens, G, P, it); it += 1
        assert ens.last_update_route == "dense"
        times = {"blocked": [], "dense": []}
        for _ in range(args.reps):
            for route in ("blocked", "dense"):
                set_route(ens, route)
                times[route].append(timed_update(ens, G, P, it)); it += 1
                assert ens.last_update_route == route
        # the same state for both routes: skip the hyper-update, so both condition on the same noise variances
        outs = {}
        for route in ("blocked", "dense"):
            set_route(ens, route)
            ens._precision_initialized = False
            ens.update(G, P, it)
            outs[route] = (ens.mean.clone(), ens.vars.clone())
        rel = lambda a, b: float(((a - b).abs().max() / b.abs().max()).item())
        diff_mean, diff_vars = rel(outs["blocked"][0], outs["dense"][0]), rel(outs["blocked"][1], outs["dense"][1])
        kts = {}
        for route in ("blocked", "dense"):
            set_route(ens, route)
            kts[route] = kernel_times(ens, G, P, it); it += 1
        nbt = (m + 63) // 64 * ((m + 63) // 64 + 1) // 2
        flop_pass = 2.0 * nbt * 64 * 64 * d * N
        gram_us, apply_us = kernel_us(kts["blocked"], "vo_post_gram_kernel"), kernel_us(kts["blocked"], "vo_post_apply_kernel")
        case = {"fine_mesh": "%dx%d" % (nf, nf), "d": d, "m": m, "N": N, "V": "per data point (W + %d RBF, l = 0.1)" % (m - (81 if nf == 128 else 25)),
                "max_rel_diff_mean": diff_mean, "max_rel_diff_vars": diff_vars,
                "dense_first_update_ms_incl_gamma": first_dense,
                "peak_bytes": {"blocked": int(peak_b), "dense": int(peak_d), "dense_gamma_resident_after": int(resident_d)},
                "kernels": kts, "algorithmic_gflop_per_row_pass": flop_pass / 1e9,
                "gram_tflops": flop_pass / gram_us / 1e6 if gram_us else None,
                "apply_tflops": flop_pass / apply_us / 1e6 if apply_us else None}
        for route, tt in times.items():
            tt = np.array(tt)
            case[route] = {"event_ms_median": float(np.median(tt)), "event_ms_min": float(tt.min())}
        case["speedup_median"] = case["dense"]["event_ms_median"] / case["blocked"]["event_ms_median"]
        result["cases"].append(case)
        print("%s m=%d N=%d  blocked %.2f ms (gram %.0f us %.1f TF/s, factor %.0f us, apply %.0f us %.1f TF/s, moments %.0f us)"
              "  dense %.2f ms (first %.1f ms)  x%.2f  peak %.0f / %.0f MB  diff %.1e / %.1e"
              % (case["fine_mesh"], m, N, case["blocked"]["event_ms_median"], gram_us, case["gram_tflops"] or 0,
                 kernel_us(kts["blocked"], "vo_post_factor_kernel"), apply_us, case["apply_tflops"] or 0,
                 kernel_us(kts["blocked"], "vo_moments_panel_kernel"), case["dense"]["event_ms_median"], first_dense,
                 case["speedup_median"], peak_b / 1e6, peak_d / 1e6, diff_mean, diff_vars), flush=True)
        del ens, outs
        torch.cuda.empty_cache()
    print("%s, power limit %s" % (result["gpu"]["name"], result["gpu"]["power_limit"]))
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r3_vo_posterior_blocked.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()

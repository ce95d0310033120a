"""Times the residual family with one weighting matrix per sample (VoPlan.residual / residual_T / residual_grad with V
[B,d,m] -> gpde_vo_residual_*, gpde_vo_residual_T_*, gpde_vo_residual_grad_* with v_stride = d*m, csrc/vo_vb.cuh)
against the same quantities through torch.bmm on the same rho and V.

    python profiles/tools/time_vo_residual_vb.py --out DIR [--reps R] [--warmup W]

Cases: config 2 (64 x 64 fine mesh, B = 4096, m = 25) and config 3 (128 x 128, N = 128, m = 256: the CGR columns plus
175 RBF columns), each in FP64 and FP32 I/O, with a pixel-input and a per-cell-input plan; log-conductivity input.  V
alone is 3.35 GB (config 2, FP64) and 4.29 GB (config 3, FP64), far beyond the 126 MB L2.  Per case:
  * CUDA-event medians over R alternated repeats (after W warm-up calls) of each new call and of its torch counterpart:
    residual against the rho-only residual call + torch.bmm(rho[B,1,d], V), residual_T against torch.bmm(V, s[B,m,1])
    + the rho-only call on w without load and Dirichlet values (= K_ff w), residual_grad alone, and the two bmm
    products alone;
  * the device time of every kernel of each new call from one torch.profiler run of its own (R calls);
  * the largest per-sample relative difference between the new calls and the torch counterparts;
  * algorithmic bytes: V plus the call's own inputs and outputs (residual: a, y, g, r; residual_T: a, s, q; gradient:
    a, y, g, gbar, grad_a), at the I/O element size, over the call time, as a fraction of 6438.8 GB/s (the copy
    bandwidth measured on the B200).
Writes DIR/r3_vo_residual_vb_cfg<k>.json with the card name and power limit."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import gpde_b200  # noqa: E402,F401
from gpde_b200 import fem  # noqa: E402
from gpde_b200.physics import LinearEllipticPhysics  # noqa: E402
from gpde_b200.VirtualObservables import VoPlan  # noqa: E402

PEAK_GBS = 6438.8


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def event_time(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def timed(fns, reps, warmup):
    """Median ms of each callable over ``reps`` alternated repeats."""
    for _ in range(warmup):
        for f in fns.values():
            f()
    torch.cuda.synchronize()
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            ts[k].append(event_time(f))
    return {k: float(np.median(v)) for k, v in ts.items()}


def kernel_times(fn, reps):
    """{kernel name: device us per call} from one torch.profiler run of ``reps`` calls."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            out[e.name] = out.get(e.name, 0.0) + e.device_time / reps
    return {k: round(v, 2) for k, v in sorted(out.items(), key=lambda kv: -kv[1])}


def rel(got, want):
    got, want = got.double(), want.double()
    scale = want.abs().amax(dim=1).clamp_min(1e-300)
    return float(((got - want).abs().amax(dim=1) / scale).max())


def run_case(nx, B, m, pixel, dtype, reps, warmup, dev):
    mesh = fem.P1Mesh(nx, nx, "right")
    fom = LinearEllipticPhysics("fom", "NDP", mesh)
    plan = VoPlan(fom, dev, mesh.pixel_of_cell(), nx * nx) if pixel else VoPlan(fom, dev)
    d, n_in, n_bc = plan.d, plan.n_inputs, plan.n_bc
    gen = torch.Generator(device=dev)
    gen.manual_seed(nx * 1000 + m)
    R = lambda *shape: torch.randn(*shape, generator=gen, device=dev, dtype=torch.float64).to(dtype)
    x, y, g, s = 0.6 * R(B, n_in), R(B, d), 0.3 * R(B, n_bc), R(B, m)
    V = R(B, d, m)
    V.mul_(d ** -0.5)
    es = 8 if dtype == torch.float64 else 4

    def torch_residual():
        _, rho = plan.residual(x, y, g, None)
        return torch.bmm(rho.unsqueeze(1), V).squeeze(1)

    def torch_residual_T():
        w = torch.bmm(V, s.unsqueeze(2)).squeeze(2)
        return plan.residual(x, w, None, None, ignore_load=True)[1]

    calls = {
        "residual": lambda: plan.residual(x, y, g, V),
        "residual_torch_bmm": torch_residual,
        "residual_T": lambda: plan.residual_T(x, V, s),
        "residual_T_torch_bmm": torch_residual_T,
        "residual_grad": lambda: plan.residual_grad(x, y, g, V, s),
        "bmm_contraction_alone": lambda: torch.bmm(y.unsqueeze(1), V),
        "bmm_expansion_alone": lambda: torch.bmm(V, s.unsqueeze(2)),
    }
    diffs = {"residual_vs_torch": rel(calls["residual"](), torch_residual()),
             "residual_T_vs_torch": rel(calls["residual_T"](), torch_residual_T())}
    t = timed(calls, reps, warmup)
    vb = B * d * m * es
    nbytes = {"residual": vb + es * B * (n_in + d + n_bc + m),
              "residual_T": vb + es * B * (n_in + m + d),
              "residual_grad": vb + es * B * (n_in + d + n_bc + m + n_in)}
    res = {"mesh": "%d x %d" % (nx, nx), "plan": "pixel" if pixel else "per-cell", "dtype": str(dtype).split(".")[-1],
           "B": B, "d": d, "m": m, "n_inputs": n_in, "V_bytes": vb, "ms": {k: round(v, 4) for k, v in t.items()},
           "algorithmic_bytes": nbytes, "max_rel_diff": diffs}
    res["fraction_of_6438.8_GBs"] = {k: round(nbytes[k] / (t[k] * 1e-3) / 1e9 / PEAK_GBS, 3) for k in nbytes}
    res["floor_ms_V_only"] = round(vb / (PEAK_GBS * 1e9) * 1e3, 4)
    res["kernels_us_per_call"] = {k: kernel_times(calls[k], reps) for k in ("residual", "residual_T", "residual_grad",
                                                                              "residual_torch_bmm", "residual_T_torch_bmm")}
    del V
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_vo_residual_vb.py measures on a CUDA device; none found")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    for cfg, (nx, B, m) in ((2, (64, 4096, 25)), (3, (128, 128, 256))):
        cases = []
        for dtype in (torch.float64, torch.float32):
            for pixel in (True, False):
                c = run_case(nx, B, m, pixel, dtype, args.reps, args.warmup, dev)
                print(json.dumps({k: c[k] for k in ("mesh", "plan", "dtype", "ms", "fraction_of_6438.8_GBs",
                                                    "max_rel_diff")}), flush=True)
                cases.append(c)
        with open(os.path.join(args.out, "r3_vo_residual_vb_cfg%d.json" % cfg), "w") as fh:
            json.dump({"gpu": info, "config": cfg, "reps": args.reps, "warmup": args.warmup, "cases": cases}, fh, indent=1)


if __name__ == "__main__":
    main()

"""Times the virtual-observable residual gradient (VoPlan.residual_grad -> gpde_vo_residual_grad_*: w = gbar_r V^T, then
grad_a by vo_grad_grid_kernel / vo_grad_cells_kernel and grad_g by vo_grad_g_kernel) on the meshes of BASELINE configs 2
and 3, with the forward residual at the same shape and a torch-ops formulation of the same gradient for comparison.

    python profiles/tools/time_vo_grad.py --out DIR [--reps R] [--warmup W]

Cases: config 2 (64 x 64 fine mesh, B = 4096, m = 25) in FP64 and FP32, pixel-input and per-cell-input plans, log and
conductivity input; config 3 (128 x 128, B = 16384, m = 256) in FP64 with a pixel-input plan.  Inputs are seeded random
fields, so the working sets exceed the 126 MB L2 except where noted by the byte counts.  Per case: CUDA-event medians
over R alternated repeats of the gradient call, the forward residual and the torch formulation; each kernel's device time
from one torch.profiler run of its own; the largest per-sample relative difference between the kernels and the torch
formulation; and bytes over time against the copy bandwidth measured in the same run.  Algorithmic bytes per sample are
s (d + n_bc + m + P) for conductivity input and s P more for log input (s = bytes per element, V counted once per
batch).  s is 8 for FP64 and 4 for FP32 I/O, so an FP32 fraction counts the bytes FP32 I/O actually moves; the same count
at 8 bytes per element is reported beside it.  The implementation adds 16 d for w = gbar_r V^T written and read back in
FP64.  Per kernel: the expansion moves s m + 8 d per sample (V once), the grad_a kernel s d + 8 d + s n_bc + s P (+ s P
for log input), vo_grad_g_kernel about (2 s + 8) n_bc (grad_g, and one w value and one input per Dirichlet dof).  Writes DIR/r3_vo_grad_<case>.json
and DIR/r3_vo_grad_summary.json with the card name and power limit."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import gpde_b200  # noqa: E402,F401
from gpde_b200.physics import setup_physics  # noqa: E402
from gpde_b200.VirtualObservables import VoPlan  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def copy_bandwidth(dev, reps=20):
    """Device-to-device copy of 2 GiB: bytes read + written over the median time (GB/s)."""
    src = torch.empty(2 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    ts = []
    for _ in range(reps + 3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dst.copy_(src)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return 2 * src.numel() / (np.median(ts[3:]) * 1e-3) / 1e9


class TorchGrad(object):
    """The same gradient from torch ops: w = gbar V^T, per-cell w~^T K_c u~ gathered and index_add'ed to the inputs,
    K_cf(a) w~ by an index_add over the cells."""

    def __init__(self, fom, c2i, dev, dtype):
        mesh = fom.mesh
        self.cells = torch.tensor(mesh.cells, device=dev)
        self.Ke = torch.tensor(mesh.element_stiffness(), device=dev, dtype=dtype)
        self.c2i = torch.tensor(c2i, device=dev)
        self.free = torch.tensor(fom.free_dofs, device=dev)
        self.bc = torch.tensor(fom.constrained_dofs, device=dev)
        self.N, self.P = mesh.num_nodes, int(self.c2i.max()) + 1

    def __call__(self, a, y, g, V, gbar, a_is_log):
        B = gbar.shape[0]
        w = torch.zeros(B, self.N, dtype=y.dtype, device=y.device)
        w[:, self.free] = gbar @ V.T
        u = torch.zeros_like(w)
        u[:, self.free], u[:, self.bc] = y, g
        wc, uc = w[:, self.cells], u[:, self.cells]
        val = (wc * torch.einsum("eij,bej->bei", self.Ke, uc)).sum(-1)
        cond = torch.exp(a) if a_is_log else a
        grad_a = torch.zeros(B, self.P, dtype=y.dtype, device=y.device).index_add_(1, self.c2i, val)
        if a_is_log:
            grad_a = grad_a * cond
        Kw = torch.einsum("eij,bej->bei", self.Ke, wc) * cond[:, self.c2i, None]
        full = torch.zeros_like(w).index_add_(1, self.cells.reshape(-1), Kw.reshape(B, -1))
        return grad_a, full[:, self.bc]


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def kernel_times(fn):
    """Device time (us) per kernel name of one call, from a torch.profiler run of its own."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith(("Memcpy", "Memset")):
            name = e.name.split("<")[0].split("(")[0].replace("void ", "").replace("gpde::", "")
            out[name] = out.get(name, 0.0) + e.time_range.elapsed_us()
    return out


def per_sample_rel(got, want):
    scale = want.abs().amax(dim=1).clamp_min(1e-300)
    return float(((got - want).abs().amax(dim=1) / scale).max())


def run_case(name, fom, pixel, dtype, a_is_log, B, m, dev, bw, args):
    mesh = fom.mesh
    c2i = mesh.pixel_of_cell() if pixel else np.arange(mesh.num_cells)
    plan = VoPlan.cached(fom, dev, pixel_input=pixel)
    gen = torch.Generator(device=dev).manual_seed(0)
    rn = lambda *s: torch.randn(*s, generator=gen, device=dev, dtype=torch.float64)
    x = 0.8 * rn(B, plan.n_inputs)
    a = (x if a_is_log else torch.exp(x)).to(dtype)
    y, g = rn(B, plan.d).to(dtype), rn(B, plan.n_bc).to(dtype)
    V, gbar = (rn(plan.d, m) / plan.d ** 0.5).to(dtype), rn(B, m).to(dtype)
    ref = TorchGrad(fom, c2i, dev, dtype)
    calls = {
        "grad": lambda: plan.residual_grad(a, y, g, V, gbar, a_is_log=a_is_log, want_grad_g=True),
        "forward_residual": lambda: plan.residual(a, y, g, V, a_is_log=a_is_log),
        "torch_ops_grad": lambda: ref(a, y, g, V, gbar, a_is_log),
    }
    ga, gg = calls["grad"]()
    ta, tg = calls["torch_ops_grad"]()
    diff = {"grad_a": per_sample_rel(ga.double(), ta.double()), "grad_g": per_sample_rel(gg.double(), tg.double())}
    times = {k: [] for k in calls}
    for rep in range(args.warmup + args.reps):
        for k, fn in calls.items():   # alternated
            t = event_ms(fn)
            if rep >= args.warmup:
                times[k].append(t)
    kernels = kernel_times(calls["grad"])
    s = torch.finfo(dtype).bits // 8
    d, n_bc, P = plan.d, plan.n_bc, plan.n_inputs
    alg = B * s * (d + n_bc + m + P + (P if a_is_log else 0)) + s * d * m
    alg8 = alg // s * 8   # the same count at 8 bytes per element whatever the I/O type
    impl = alg + B * 16 * d
    med = {k: float(np.median(v)) for k, v in times.items()}
    kernel_bytes = {   # implementation bytes each kernel moves (w in FP64)
        "expand": B * (s * m + 8 * d) + s * d * m,
        "grad_a": B * (s * d + 8 * d + s * n_bc + s * P + (s * P if a_is_log else 0)),
        # grad_g written, plus (about) one FP64 w value and one input per Dirichlet dof: the free column and the cells
        # next to the boundary
        "grad_g": B * (s + 8 + s) * n_bc,
    }
    kern = {}
    for kname, us in kernels.items():
        kind = "grad_a" if kname in ("vo_grad_grid_kernel", "vo_grad_cells_kernel") else (
            "grad_g" if kname == "vo_grad_g_kernel" else (
                "expand" if kname in ("vo_expand_dmma_kernel", "vo_expand_kernel", "vo_gemm_kernel") else None))
        entry = {"us": us}
        if kind:
            entry["bytes"] = kernel_bytes[kind]
            entry["fraction_of_copy_bandwidth"] = kernel_bytes[kind] / (us * 1e-6) / 1e9 / bw
        kern[kname] = entry
    res = {"case": name, "B": B, "m": m, "d": d, "n_bc": n_bc, "n_inputs": P, "dtype": str(dtype).replace("torch.", ""),
           "plan": "pixel" if pixel else "per-cell", "input": "log" if a_is_log else "conductivity",
           "median_ms": med, "kernels_us": kern, "max_per_sample_rel_diff_vs_torch": diff,
           "algorithmic_bytes": alg, "algorithmic_bytes_at_8_bytes_per_element": alg8, "implementation_bytes": impl,
           "grad_fraction_of_copy_bandwidth_algorithmic": alg / (med["grad"] * 1e-3) / 1e9 / bw,
           "grad_fraction_of_copy_bandwidth_algorithmic_at_8_bytes_per_element": alg8 / (med["grad"] * 1e-3) / 1e9 / bw,
           "grad_fraction_of_copy_bandwidth_implementation": impl / (med["grad"] * 1e-3) / 1e9 / bw,
           "speedup_vs_torch_ops": med["torch_ops_grad"] / med["grad"]}
    print("%-28s grad %.3f ms (alg %.0f%% / impl %.0f%% of copy BW)  forward %.3f ms  torch %.3f ms  kernels %s  diff %.1e/%.1e"
          % (name, med["grad"], 100 * res["grad_fraction_of_copy_bandwidth_algorithmic"],
             100 * res["grad_fraction_of_copy_bandwidth_implementation"], med["forward_residual"], med["torch_ops_grad"],
             {k: round(v["us"], 1) for k, v in kern.items()}, diff["grad_a"], diff["grad_g"]), flush=True)
    with open(os.path.join(args.out, "r3_vo_grad_%s.json" % name), "w") as f:
        json.dump(res, f, indent=1)
    del calls, ref
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    bw = copy_bandwidth(dev)
    print("%s, power limit %s, copy bandwidth %.0f GB/s" % (info["name"], info["power_limit"], bw), flush=True)
    cases = []
    fom2 = setup_physics(4, 4, 4, "ND")["fom"]
    for dtype in (torch.float64, torch.float32):
        for pixel in (True, False):
            for a_is_log in (True, False):
                name = "cfg2_%s_%s_%s" % ("f64" if dtype == torch.float64 else "f32", "pixel" if pixel else "cell",
                                          "log" if a_is_log else "cond")
                cases.append(run_case(name, fom2, pixel, dtype, a_is_log, 4096, 25, dev, bw, args))
    fom3 = setup_physics(8, 8, 4, "ND")["fom"]
    cases.append(run_case("cfg3_f64_pixel_log", fom3, True, torch.float64, True, 16384, 256, dev, bw, args))
    with open(os.path.join(args.out, "r3_vo_grad_summary.json"), "w") as f:
        json.dump({"gpu": info, "copy_bandwidth_GBps": bw, "reps": args.reps, "warmup": args.warmup, "cases": cases}, f,
                  indent=1)


if __name__ == "__main__":
    main()

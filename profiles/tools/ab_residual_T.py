"""A/B on ONE box: the transposed application q = K_ff(a) (V s) in one kernel (WT variant of vo_grid2_kernel) against the
two-kernel route (GPDE_VO_FUSED_T=0: expansion kernel, w [B,d] through HBM, marching kernel); device time per call from
CUDA-graph replays, three rounds, FP64 / FP32 I/O, conductivity / log input.
    python profiles/tools/ab_residual_T.py [workload] [B]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
import gpde_b200  # noqa
from gpde_b200.VirtualObservables import VoPlan
from gpde_b200.workloads import Workload
name = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
B = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
extra = [dict(kv.split("=") for kv in spec.split(",")) for spec in sys.argv[3:]]   # e.g. GPDE_GRID2_SPC=24
dev = torch.device("cuda", 0)
w = Workload(name, B=min(B, 4096), seed=0)
base = VoPlan.cached(w.physics["fom"], dev, pixel_input=True)
T = lambda t: torch.tensor(t, device=dev)
rep = (B + w.B - 1) // w.B
a_log = T(w.log_image).repeat(rep, 1)[:B].contiguous()
a, V = torch.exp(a_log), T(w.V)
s = torch.randn(B, w.m, dtype=torch.float64, device=dev)
plans = {"one kernel": base, "two kernels": base.variant(GPDE_VO_FUSED_T="0")}
for e in extra:
    plans["one kernel " + ",".join("%s=%s" % (k[5:], v) for k, v in e.items())] = base.variant(**e)
ref = plans["two kernels"].residual_T(a, V, s, a_is_log=False)
err = (plans["one kernel"].residual_T(a, V, s, a_is_log=False) - ref).abs().max() / ref.abs().max()
print("B %d m %d: one kernel vs two kernels rel err %.2e" % (B, w.m, err.item()))

def timed(plan, log, f32=False):
    c = (lambda t: t.float()) if f32 else (lambda t: t)
    aa, VV, ss = c(a_log if log else a), c(V), c(s)
    fn = lambda: plan.residual_T(aa, VV, ss, a_is_log=log)
    for _ in range(3): fn()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            keep = [fn() for _ in range(10)]
    gr.replay(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): gr.replay()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 50 * 1e3

for rnd in range(3):
    for label, p in plans.items():
        print("round %d %-28s: conductivity %.2f us, log input %.2f us, FP32 I/O %.2f us" %
              (rnd, label, timed(p, False), timed(p, True), timed(p, False, True)), flush=True)

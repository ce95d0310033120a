"""VO residual at cfg2 with and without the in-kernel exp (a_is_log), and for m = 8 / 16 / 25: how the kernel time
responds to removing instruction classes (a diagnostic for what bounds vo_grid2_kernel)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
import gpde_b200  # noqa
from gpde_b200.VirtualObservables import VoPlan
from gpde_b200.workloads import Workload

w = Workload("cfg2", seed=0)
dev = torch.device("cuda", 0)
plan = VoPlan.cached(w.physics["fom"], dev, pixel_input=True)
a = torch.tensor(w.log_image, device=dev)
ea = torch.exp(a)
y = torch.tensor(w.y, device=dev)
g = torch.tensor(w.g_fom[0], device=dev)
V = torch.tensor(w.V, device=dev)


def t(fn, n=30):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3

print("m=25 log input      : %.1f us" % t(lambda: plan.residual(a, y, g, V)))
print("m=25 conductivities : %.1f us" % t(lambda: plan.residual(ea, y, g, V, a_is_log=False)))
for m in (16, 8):
    Vm = V[:, :m].contiguous()
    print("m=%-2d log input      : %.1f us" % (m, t(lambda: plan.residual(a, y, g, Vm))))
    print("m=%-2d conductivities : %.1f us" % (m, t(lambda: plan.residual(ea, y, g, Vm, a_is_log=False))))

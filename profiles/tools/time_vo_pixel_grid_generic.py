"""Device time of the VO residual and residual_T on a pixel grid the structured-grid kernel does not serve (width 66, not
one of 16 / 32 / 64 / 128): such plans take the generic kernels (vo_fused.cuh for m <= 32, version 1 otherwise).  No
bench.py workload reaches this case.  CUDA events around 50 calls after 5 warm-up calls; at the default size a and y are
143 MB each, more than the 126 MB of L2.
    python profiles/tools/time_vo_pixel_grid_generic.py [nx] [B] [m]"""
import os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np
import torch
import gpde_b200  # noqa
from gpde_b200 import fem
from gpde_b200.physics import LinearEllipticPhysics
from gpde_b200.VirtualObservables import VoPlan

nx = int(sys.argv[1]) if len(sys.argv) > 1 else 66
B = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
m = int(sys.argv[3]) if len(sys.argv) > 3 else 25
dev = torch.device("cuda", 0)
mesh = fem.P1Mesh(nx, nx, "right")
fom = LinearEllipticPhysics("fom", "ND", mesh)
plan = VoPlan(fom, dev, mesh.pixel_of_cell(), nx * nx)
rng = np.random.RandomState(0)
bc = mesh.dirichlet_dofs()[0]
T = lambda t: torch.tensor(t, device=dev)
a_log = T(rng.normal(0.4, 0.8, size=(B, nx * nx)))
a = torch.exp(a_log)
y, g = T(rng.normal(size=(B, fom.dim_out))), T(rng.uniform(-0.5, 0.5, size=(B, bc.size)))
V, s = T(rng.normal(size=(fom.dim_out, m))), T(rng.normal(size=(B, m)))


def timed(fn, n=50):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print("%s | %dx%d pixel grid, B %d, m %d, kernel_path %d" % (card, nx, nx, B, m, plan.kernel_path(m)))
for rnd in range(3):
    print("round %d: residual log input %.1f us, conductivity input %.1f us, residual_T %.1f us" %
          (rnd, timed(lambda: plan.residual(a_log, y, g, V)), timed(lambda: plan.residual(a, y, g, V, a_is_log=False)),
           timed(lambda: plan.residual_T(a_log, V, s))), flush=True)

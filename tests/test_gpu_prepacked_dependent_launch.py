"""With prepacked weights the structured-grid residual kernel is launched as a programmatic dependent of whatever the
stream ran before it (vo.cu, launch_grid2).  It must wait for that work before it reads a, y or g: inputs rewritten in
place by the kernel right before the call are the ones the residual sees."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_inputs_written_just_before_a_prepacked_call(dtype, dev):
    from gpde_b200 import fem
    from gpde_b200.physics import LinearEllipticPhysics
    from gpde_b200.VirtualObservables import VoPlan
    nx, B = 64, 4096
    rng = np.random.RandomState(11)
    mesh = fem.P1Mesh(nx, nx, "right")
    fom = LinearEllipticPhysics("fom", "NDP", mesh)
    plan = VoPlan(fom, dev, mesh.pixel_of_cell(), nx * nx)
    T = lambda t: torch.tensor(t, dtype=dtype, device=dev)
    a = T(rng.normal(0.4, 0.8, size=(B, nx * nx)))
    y = T(rng.normal(size=(B, fom.dim_out)))
    g = T(rng.uniform(-0.5, 0.5, size=(B, mesh.dirichlet_dofs()[0].size)))
    V = T(rng.normal(size=(fom.dim_out, 25)))
    pw = plan.pack_weights(V, B)
    a_buf, y_buf, g_buf = torch.zeros_like(a), torch.zeros_like(y), torch.zeros_like(g)
    torch.cuda.synchronize(dev)
    for k in range(4):
        s = 1.0 + 0.25 * k
        # in-place writes by kernels of the same stream, immediately followed by the prepacked call
        torch.mul(a, s, out=a_buf)
        torch.mul(y, s, out=y_buf)
        torch.mul(g, s, out=g_buf)
        r = plan.residual(a_buf, y_buf, g_buf, pw)
        want = plan.residual(a * s, y * s, g * s, V)
        assert torch.equal(r, want), k

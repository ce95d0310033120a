"""Gradient of the virtual-observable residual in the conductivity input and the Dirichlet values
(gpde_vo_residual_grad_*, csrc/vo_grad.cuh) against an independent float64 torch reference built on the CPU from
oracle/fem_p1 with autograd, against the exact identities that follow from linearity, and through VoResidualFn."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import fem_p1

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


_PLANS = {}


def _problem(nx, ny, diagonal, pixel, dev):
    """(plan, oracle data) for a pixel-input or per-cell-input plan of the nx x ny mesh; plans are cached."""
    key = (nx, ny, diagonal, pixel)
    if key not in _PLANS:
        from gpde_b200 import fem
        from gpde_b200.physics import LinearEllipticPhysics
        from gpde_b200.VirtualObservables import VoPlan
        mesh = fem.P1Mesh(nx, ny, diagonal)
        fom = LinearEllipticPhysics("fom", "NDP", mesh)
        coords, cells = fem_p1.unit_square_mesh(nx, ny, diagonal)
        assert np.array_equal(cells, mesh.cells)
        bc, _, free = fem_p1.dirichlet_left_right(coords, "NDP", np.zeros(4))
        c2i = fem_p1.pixel_of_cell(coords, cells, nx, ny) if pixel else np.arange(len(cells))
        plan = VoPlan(fom, dev, c2i, nx * ny) if pixel else VoPlan(fom, dev)
        ref = dict(coords=coords, cells=torch.tensor(cells), Ke=torch.tensor(fem_p1.element_stiffness_all(coords, cells)),
                   c2i=torch.tensor(c2i), bc=torch.tensor(bc), free=torch.tensor(free), n_nodes=len(coords))
        _PLANS[key] = (plan, ref)
    return _PLANS[key]


def _ref_residual(ref, inp, a_is_log, y, g, V):
    """r [B,m] = V^T (K(a) u~)_free in float64 torch on the CPU (index_add assembly, differentiable in every input)."""
    a_cell = (torch.exp(inp) if a_is_log else inp)[:, ref["c2i"]]             # [B,E]
    B = inp.shape[0]
    u = torch.zeros(B, ref["n_nodes"], dtype=torch.float64)
    u = u.index_copy(1, ref["free"], y).index_copy(1, ref["bc"], g)
    uc = u[:, ref["cells"]]                                                    # [B,E,3]
    Ku = torch.einsum("eij,bej->bei", ref["Ke"], uc) * a_cell[..., None]
    full = torch.zeros(B, ref["n_nodes"], dtype=torch.float64).index_add(1, ref["cells"].reshape(-1), Ku.reshape(B, -1))
    return full[:, ref["free"]] @ V


def _ref_grads(ref, inp, a_is_log, y, g, V, gbar):
    inp, g = inp.clone().requires_grad_(True), g.clone().requires_grad_(True)
    (_ref_residual(ref, inp, a_is_log, y, g, V) * gbar).sum().backward()
    return inp.grad, g.grad


def _inputs(plan, ref, B, m, kind, seed):
    """Per-sample inputs on the CPU in float64: log field x, y, Dirichlet values g (ND or NDP), V, gbar_r."""
    rng = np.random.RandomState(seed)
    x = 0.6 * rng.standard_normal((B, plan.n_inputs))
    y = rng.standard_normal((B, plan.d))
    if kind == "ND":
        g = np.stack([fem_p1.dirichlet_left_right(ref["coords"], "ND")[1]] * B)
    else:
        g = np.stack([fem_p1.dirichlet_left_right(ref["coords"], "NDP", u)[1] for u in rng.uniform(-0.5, 0.5, (B, 4))])
    V = rng.standard_normal((plan.d, m)) / np.sqrt(plan.d)
    gbar = rng.standard_normal((B, m))
    return [torch.tensor(t) for t in (x, y, g, V, gbar)]


def _per_sample_rel(got, want):
    got, want = got.double().cpu(), want.double().cpu()
    scale = want.abs().amax(dim=1).clamp_min(1e-300)
    return float(((got - want).abs().amax(dim=1) / scale).max())


def _grad_kernels(fn):
    """Names of the vo_grad_* kernels fn launches (torch.profiler).  fn launches at least the expansion kernel, so a capture
    without any of the project's kernels has lost its device records (in a long test process the profiler sometimes returns
    a short capture empty) and is taken again."""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        seen = [e.name for e in prof.events()]
        if any("gpde::" in s for s in seen):
            break
    return {k for k in ("vo_grad_grid_kernel", "vo_grad_cells_kernel", "vo_grad_g_kernel") if any(k in s for s in seen)}


def _call(plan, inp, y, g, V, gbar, dev, a_is_log, dtype=torch.float64, **kw):
    cast = lambda t: None if t is None else t.to(device=dev, dtype=dtype)
    return plan.residual_grad(cast(inp if a_is_log else torch.exp(inp)), cast(y), cast(g), cast(V), cast(gbar),
                              a_is_log=a_is_log, **kw)


@pytest.mark.parametrize("pixel", [True, False])
@pytest.mark.parametrize("diagonal", ["right", "alternating"])
@pytest.mark.parametrize("shape", [(16, 16), (32, 32), (64, 64), (8, 6), (16, 8), (32, 16)])
def test_grad_against_torch_reference(shape, diagonal, pixel, dev):
    plan, ref = _problem(shape[0], shape[1], diagonal, pixel, dev)
    B = 3
    for m in (1, 4, 25, 32, 33, 64):
        for kind in ("ND", "NDP"):
            x, y, g, V, gbar = _inputs(plan, ref, B, m, kind, seed=m)
            for a_is_log in (True, False):
                inp = x if a_is_log else torch.exp(x)
                want_a, want_g = _ref_grads(ref, inp, a_is_log, y, g, V, gbar)
                ga, gg = _call(plan, x, y, g, V, gbar, dev, a_is_log, want_grad_g=True)
                assert _per_sample_rel(ga, want_a) < 1e-10, (m, kind, a_is_log)
                assert _per_sample_rel(gg, want_g) < 1e-10, (m, kind, a_is_log)


def test_pixel_route_matches_cell_route(dev):
    """The marching kernel (pixel plan) against the per-cell kernel: grad[p] = grad[c1] + grad[c2]."""
    for diagonal in ("right", "alternating"):
        pix, ref = _problem(16, 16, diagonal, True, dev)
        cel, _ = _problem(16, 16, diagonal, False, dev)
        x, y, g, V, gbar = _inputs(pix, ref, 64, 25, "NDP", seed=1)
        xc = x[:, ref["c2i"]]
        for a_is_log in (True, False):
            assert _grad_kernels(lambda: _call(pix, x, y, g, V, gbar, dev, a_is_log)) == {"vo_grad_grid_kernel"}
            assert _grad_kernels(lambda: _call(cel, xc, y, g, V, gbar, dev, a_is_log)) == {"vo_grad_cells_kernel"}
            gp, _ = _call(pix, x, y, g, V, gbar, dev, a_is_log)
            gc, _ = _call(cel, xc, y, g, V, gbar, dev, a_is_log)
            summed = torch.zeros_like(gp).index_add_(1, ref["c2i"].to(dev), gc)
            assert _per_sample_rel(gp, summed) < 1e-12
    # rectangular pixels (horizontal and vertical couplings differ): the marching kernel pairs each with its edges
    for shape in ((16, 8), (32, 16)):
        pix, ref = _problem(shape[0], shape[1], "right", True, dev)
        cel, _ = _problem(shape[0], shape[1], "right", False, dev)
        x, y, g, V, gbar = _inputs(pix, ref, 16, 25, "NDP", seed=3)
        assert _grad_kernels(lambda: _call(pix, x, y, g, V, gbar, dev, True)) == {"vo_grad_grid_kernel"}
        gp, _ = _call(pix, x, y, g, V, gbar, dev, True)
        gc, _ = _call(cel, x[:, ref["c2i"]], y, g, V, gbar, dev, True)
        assert _per_sample_rel(gp, torch.zeros_like(gp).index_add_(1, ref["c2i"].to(dev), gc)) < 1e-12
    # an 8 x 6 pixel plan is not a lean-grid mesh: the per-cell kernel serves it
    pix, ref = _problem(8, 6, "right", True, dev)
    x, y, g, V, gbar = _inputs(pix, ref, 4, 4, "ND", seed=2)
    assert _grad_kernels(lambda: _call(pix, x, y, g, V, gbar, dev, True, want_grad_g=True)) == \
        {"vo_grad_cells_kernel", "vo_grad_g_kernel"}


@pytest.mark.parametrize("cfg", ["cfg2", "cfg3"])
def test_linearity_identities_at_full_size(cfg, dev):
    """<grad_a, d> = gbar.(r(a+d) - r(a)), <grad_g, d> = gbar.(r(g+d) - r(g)), sum_p a_p grad_a[p] = gbar.r, per sample,
    against the existing residual kernels (no load vector)."""
    from gpde_b200.physics import setup_physics
    from gpde_b200.VirtualObservables import VoPlan
    nx, B, m = (4, 4096, 25) if cfg == "cfg2" else (8, 2048, 256)
    fom = setup_physics(nx, nx, 4, "ND")["fom"]
    plan = VoPlan.cached(fom, dev, pixel_input=True)
    gen = torch.Generator(device=dev).manual_seed(7)
    rn = lambda *s: torch.randn(*s, generator=gen, device=dev, dtype=torch.float64)
    a = torch.exp(0.6 * rn(B, plan.n_inputs))
    y, g = rn(B, plan.d), rn(B, plan.n_bc)
    V, gbar = rn(plan.d, m) / plan.d ** 0.5, rn(B, m)
    da, dg = 0.3 * a * rn(B, plan.n_inputs), rn(B, plan.n_bc)
    ga, gg = plan.residual_grad(a, y, g, V, gbar, a_is_log=False, want_grad_g=True)
    r0 = plan.residual(a, y, g, V, a_is_log=False)

    def check(lhs_terms, dr):
        lhs, rhs_terms = lhs_terms.sum(1), gbar * dr
        scale = torch.maximum(lhs_terms.abs().sum(1), rhs_terms.abs().sum(1))
        assert float(((lhs - rhs_terms.sum(1)).abs() / scale).max()) < 1e-10

    check(ga * da, plan.residual(a + da, y, g, V, a_is_log=False) - r0)
    check(gg * dg, plan.residual(a, y, g + dg, V, a_is_log=False) - r0)
    check(a * ga, r0)
    gx, _ = plan.residual_grad(torch.log(a), y, g, V, gbar, a_is_log=True)
    assert _per_sample_rel(gx, a * ga) < 1e-12


def test_gradcheck_through_autograd(dev):
    from gpde_b200 import fem
    from gpde_b200.physics import LinearEllipticPhysics
    from gpde_b200.VirtualObservables import VoPlan, VoResidualFn
    fom = LinearEllipticPhysics("fom", "NDP", fem.P1Mesh(4, 4))
    plan = VoPlan(fom, dev)
    gen = torch.Generator(device=dev).manual_seed(3)
    rn = lambda *s: torch.randn(*s, generator=gen, device=dev, dtype=torch.float64)
    B, m = 3, 5
    y = rn(B, plan.d).requires_grad_(True)
    x = (0.5 * rn(B, plan.n_inputs)).requires_grad_(True)
    g = rn(B, plan.n_bc).requires_grad_(True)
    V = rn(plan.d, m)
    assert torch.autograd.gradcheck(lambda y_, x_, g_: VoResidualFn.apply(y_, x_, g_, V, plan, True), (y, x, g))
    # a and g alone, shared across the batch (1-D), y without grad
    x1 = x[0].detach().clone().requires_grad_(True)
    g1 = g[0].detach().clone().requires_grad_(True)
    assert torch.autograd.gradcheck(lambda x_, g_: VoResidualFn.apply(y.detach(), x_, g_, V, plan, True), (x1, g1))


@pytest.mark.parametrize("pixel", [True, False])
@pytest.mark.parametrize("m", [4, 25, 64])
def test_fp32_io_matches_fp64_on_rounded_inputs(pixel, m, dev):
    plan, ref = _problem(64, 64, "right", pixel, dev)
    x, y, g, V, gbar = _inputs(plan, ref, 257, m, "NDP", seed=5)
    x, y, g, V, gbar = (t.float().double() for t in (x, y, g, V, gbar))
    for a_is_log in (True, False):
        inp = x if a_is_log else torch.exp(x).float().double()
        f32 = plan.residual_grad(*(t.to(dev, torch.float32) for t in (inp, y, g, V, gbar)), a_is_log=a_is_log,
                                 want_grad_g=True)
        f64 = plan.residual_grad(*(t.to(dev) for t in (inp, y, g, V, gbar)), a_is_log=a_is_log, want_grad_g=True)
        for lo, hi in zip(f32, f64):
            assert lo.dtype == torch.float32
            assert _per_sample_rel(lo, hi) < 2e-6


def test_edge_cases_with_one_workspace_query(dev):
    from gpde_b200 import _lib
    plan, ref = _problem(16, 16, "right", True, dev)
    x, y, g, V, gbar = (t.to(dev) for t in _inputs(plan, ref, 8, 25, "NDP", seed=9))
    full_a, full_g = plan.residual_grad(x, y, g, V, gbar, want_grad_g=True)
    # NULL outputs: the other one is unchanged, bit for bit
    assert torch.equal(plan.residual_grad(x, y, g, V, gbar)[0], full_a)
    ga, gg = plan.residual_grad(x, y, g, V, gbar, want_grad_a=False, want_grad_g=True)
    assert ga is None and torch.equal(gg, full_g)
    # y = None and g = None mean zeros
    z_a, z_g = plan.residual_grad(x, torch.zeros_like(y), torch.zeros_like(g), V, gbar, want_grad_g=True)
    n_a, n_g = plan.residual_grad(x, None, None, V, gbar, want_grad_g=True)
    assert torch.equal(z_a, n_a) and torch.equal(z_g, n_g)
    # shared a and g (stride 0): the per-sample gradients summed over the batch
    for pixel in (True, False):
        p2, r2 = _problem(16, 16, "right", pixel, dev)
        xs, ys, gs, Vs, gbs = (t.to(dev) for t in _inputs(p2, r2, 8, 25, "NDP", seed=10))
        sa, sg = p2.residual_grad(xs[0], ys, gs[0], Vs, gbs, want_grad_g=True)
        ea, eg = p2.residual_grad(xs[:1].expand(8, -1).contiguous(), ys, gs[:1].expand(8, -1).contiguous(), Vs, gbs,
                                  want_grad_g=True)
        assert sa.shape == (p2.n_inputs,) and sg.shape == (p2.n_bc,)
        assert torch.allclose(sa, ea.sum(0), rtol=1e-13, atol=0) and torch.allclose(sg, eg.sum(0), rtol=1e-13, atol=0)
    # B = 0 and B = 1
    e_a, e_g = plan.residual_grad(x[:0], y[:0], g[:0], V, gbar[:0], want_grad_g=True)
    assert e_a.shape == (0, plan.n_inputs) and e_g.shape == (0, plan.n_bc)
    o_a, o_g = plan.residual_grad(x[3:4], y[3:4], g[3:4], V, gbar[3:4], want_grad_g=True)
    assert torch.equal(o_a, full_a[3:4]) and torch.equal(o_g, full_g[3:4])
    # bitwise sample-permutation equivariance
    perm = torch.randperm(8, generator=torch.Generator().manual_seed(0)).to(dev)
    p_a, p_g = plan.residual_grad(x[perm], y[perm], g[perm], V, gbar[perm], want_grad_g=True)
    assert torch.equal(p_a, full_a[perm]) and torch.equal(p_g, full_g[perm])
    # batched arguments whose batch differs from gbar_r's: ValueError before any launch
    for bad_args in ((x[:1], y, g), (x, y[:5], g), (x, y, g[:2])):
        with pytest.raises(ValueError):
            plan.residual_grad(*bad_args, V, gbar)
    # argument errors: GpdeLibraryError, no device fault
    lib = _lib.load()
    ws = torch.empty(int(lib.gpde_vo_workspace_bytes(plan.handle, 8, 25)) + 64, dtype=torch.uint8, device=dev)
    P = lambda t: _lib.ptr(t, dev)
    st = _lib.stream_of(dev)
    Vc, gbc = V.contiguous(), gbar.contiguous()
    out_a = torch.empty(8, plan.n_inputs, dtype=torch.float64, device=dev)
    base = dict(a=P(x), a_stride=plan.n_inputs, V=P(Vc), m=25, gbar=P(gbc), ws=P(ws))
    bad = [dict(m=0), dict(m=-3), dict(gbar=None), dict(V=None), dict(a=None), dict(a_stride=7),
           dict(ws=ctypes.c_void_p(ws.data_ptr() + 8)), dict(ws=None)]
    for change in bad:
        k = dict(base, **change)
        rc = lib.gpde_vo_residual_grad_f64(plan.handle, k["a"], k["a_stride"], 1, P(y), P(g), plan.n_bc, k["V"], 0, k["m"],
                                           k["gbar"], P(out_a), None, k["ws"], 8, st)
        with pytest.raises(_lib.GpdeLibraryError):
            _lib.check(rc, "gpde_vo_residual_grad_f64")
    torch.cuda.synchronize()
    assert torch.equal(plan.residual_grad(x, y, g, V, gbar)[0], full_a)


def test_batch_that_wraps_the_grid_stride_loops(dev):
    """More outputs than the capped launch grids hold threads (cap: 8 CTAs of 256 threads per SM for the marching kernel,
    16 for the others), on both routes."""
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    for pixel in (True, False):
        plan, ref = _problem(16, 16, "right", pixel, dev)
        B = n_sm * 8 * 256 // 16 + 5
        assert B * 16 > n_sm * 8 * 256 and B * plan.n_inputs > n_sm * 16 * 256 and B * plan.n_bc > n_sm * 16 * 256
        x, y, g, V, gbar = _inputs(plan, ref, B, 4, "NDP", seed=11)
        want_a, want_g = _ref_grads(ref, x, True, y, g, V, gbar)
        ga, gg = _call(plan, x, y, g, V, gbar, dev, True, want_grad_g=True)
        assert _per_sample_rel(ga, want_a) < 1e-10 and _per_sample_rel(gg, want_g) < 1e-10

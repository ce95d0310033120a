"""The virtual-observable residual family with one weighting matrix per sample, V [B,d,m] (gpde_vo_residual_*,
gpde_vo_residual_T_*, gpde_vo_residual_grad_* with v_stride = d*m, csrc/vo_vb.cuh): against oracle/vo_ref.py per sample
with K and f from oracle/fem_p1.py, against a shared V, through VoResidualFn and through the ensemble API; and the one
workspace query of the family, for either layout."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import fem_p1, vo_ref

pytestmark = pytest.mark.gpu

GPDE_ERR_ARG = -1


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


_CASES = {}


def _case(nx, ny, pixel, load, dev):
    """(plan, oracle data) of the nx x ny mesh with pixel or per-cell conductivity input; a random load vector when
    ``load``.  Cached per configuration."""
    key = (nx, ny, pixel, load)
    if key not in _CASES:
        from gpde_b200 import fem
        from gpde_b200.physics import LinearEllipticPhysics
        from gpde_b200.VirtualObservables import VoPlan
        mesh = fem.P1Mesh(nx, ny, "right")
        fom = LinearEllipticPhysics("fom", "NDP", mesh)
        coords, cells = fem_p1.unit_square_mesh(nx, ny, "right")
        assert np.array_equal(cells, mesh.cells)
        bc, _, free = fem_p1.dirichlet_left_right(coords, "ND")
        assert np.array_equal(bc, fom.constrained_dofs) and np.array_equal(free, fom.free_dofs)
        f = np.random.RandomState(nx * 100 + ny).standard_normal(len(coords)) if load else None
        c2i = mesh.pixel_of_cell() if pixel else np.arange(len(cells))
        n_in = nx * ny if pixel else len(cells)
        plan = VoPlan(fom, dev, c2i, n_in, load=f) if pixel else VoPlan(fom, dev, load=f)
        _CASES[key] = (plan, dict(coords=coords, cells=cells, bc=bc, free=free, f=f, c2i=np.asarray(c2i)))
    return _CASES[key]


def _inputs(plan, ref, B, m, kind, seed):
    """Per-sample float64 inputs on the host: log field x [B,n_inputs], y [B,d], Dirichlet values g [B,n_bc] (ND: the
    same values for every sample, NDP: random per sample), V [B,d,m], s [B,m]."""
    rng = np.random.RandomState(seed)
    x = 0.6 * rng.standard_normal((B, plan.n_inputs))
    y = rng.standard_normal((B, plan.d))
    if kind == "ND":
        g = np.stack([fem_p1.dirichlet_left_right(ref["coords"], "ND")[1]] * B)
    else:
        g = np.stack([fem_p1.dirichlet_left_right(ref["coords"], "NDP", u)[1] for u in rng.uniform(-0.5, 0.5, (B, 4))])
    V = rng.standard_normal((B, plan.d, m)) / np.sqrt(plan.d)
    s = rng.standard_normal((B, m))
    return x, y, g, V, s


def _oracle(ref, x, y, g, V, s):
    """(r, q) per sample from vo_ref with (K_ff, f_eff) of fem_p1."""
    rs, qs = [], []
    for b in range(x.shape[0]):
        K, f = fem_p1.assemble_system_free(ref["coords"], ref["cells"], np.exp(x[b])[ref["c2i"]], ref["bc"], g[b],
                                           ref["free"], ref["f"])
        rs.append(vo_ref.vo_residual(K, f, V[b], y[b]))
        qs.append(vo_ref.vo_residual_transposed(K, V[b], s[b]))
    return np.stack(rs), np.stack(qs)


def _ref_grads(ref, x, y, g, V, gbar):
    """(d/dx, d/dg) of sum(gbar * r) with r_b = V_b^T (K(exp x_b) u~_b)_free, float64 torch autograd on the host."""
    cells, free, bc = (torch.tensor(ref[k]) for k in ("cells", "free", "bc"))
    Ke = torch.tensor(fem_p1.element_stiffness_all(ref["coords"], ref["cells"]))
    xt, gt = torch.tensor(x).requires_grad_(True), torch.tensor(g).requires_grad_(True)
    B, n = x.shape[0], len(ref["coords"])
    a_cell = torch.exp(xt)[:, torch.tensor(ref["c2i"])]
    u = torch.zeros(B, n, dtype=torch.float64).index_copy(1, free, torch.tensor(y)).index_copy(1, bc, gt)
    Ku = torch.einsum("eij,bej->bei", Ke, u[:, cells]) * a_cell[..., None]
    full = torch.zeros(B, n, dtype=torch.float64).index_add(1, cells.reshape(-1), Ku.reshape(B, -1))
    r = torch.einsum("bi,bim->bm", full[:, free], torch.tensor(V))
    (r * torch.tensor(gbar)).sum().backward()
    return xt.grad.numpy(), gt.grad.numpy()


def _rel(got, want):
    """Largest per-sample error relative to the sample's largest entry."""
    got = got.double().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    got, want = got.reshape(want.shape[0], -1), np.asarray(want).reshape(want.shape[0], -1)
    scale = np.maximum(np.abs(want).max(axis=1), 1e-300)
    return float((np.abs(got - want).max(axis=1) / scale).max())


MS = [1, 8, 25, 32, 33, 64, 100, 256]
MESHES = [(16, 8, True), (6, 5, False)]   # pixel plan (structured-grid kernels) and per-cell plan (with a load vector)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("kind", ["ND", "NDP"])
@pytest.mark.parametrize("mesh", MESHES, ids=["pixel", "cell"])
@pytest.mark.parametrize("m", MS)
def test_per_sample_calls_match_the_oracle(m, mesh, kind, dtype, dev):
    nx, ny, pixel = mesh
    plan, ref = _case(nx, ny, pixel, not pixel, dev)
    B = 5
    x, y, g, V, s = _inputs(plan, ref, B, m, kind, seed=m * 7 + nx)
    if dtype == torch.float32:   # the oracle sees the float-rounded inputs
        x, y, g, V, s = (t.astype(np.float32).astype(np.float64) for t in (x, y, g, V, s))
    T = lambda t: torch.tensor(t, dtype=dtype, device=dev)
    r_ref, q_ref = _oracle(ref, x, y, g, V, s)
    tol = 1e-10 if dtype == torch.float64 else 1e-5
    r, rho = plan.residual(T(x), T(y), T(g), T(V), want_rho=True)
    assert r.shape == (B, m) and r.dtype == dtype
    assert _rel(r, r_ref) < tol
    assert torch.equal(rho, plan.residual(T(x), T(y), T(g), None)[1])
    assert _rel(plan.residual_T(T(x), T(V), T(s)), q_ref) < tol
    ga_ref, gg_ref = _ref_grads(ref, x, y, g, V, s)
    ga, gg = plan.residual_grad(T(x), T(y), T(g), T(V), T(s), want_grad_g=True)
    assert _rel(ga, ga_ref) < tol and _rel(gg, gg_ref) < tol


@pytest.mark.parametrize("mesh", MESHES, ids=["pixel", "cell"])
@pytest.mark.parametrize("m", [8, 100])
def test_shared_field_and_dirichlet_values(m, mesh, dev):
    """a [n_inputs] and g [n_bc] shared by the batch, V per sample."""
    nx, ny, pixel = mesh
    plan, ref = _case(nx, ny, pixel, not pixel, dev)
    B = 4
    x, y, g, V, s = _inputs(plan, ref, B, m, "NDP", seed=m + 3)
    xs, gs = np.repeat(x[:1], B, axis=0), np.repeat(g[:1], B, axis=0)
    T = lambda t: torch.tensor(t, dtype=torch.float64, device=dev)
    r_ref, q_ref = _oracle(ref, xs, y, gs, V, s)
    assert _rel(plan.residual(T(x[0]), T(y), T(g[0]), T(V)), r_ref) < 1e-10
    assert _rel(plan.residual_T(T(x[0]), T(V), T(s)), q_ref) < 1e-10
    # nothing batched but V: the batch is V's
    r0_ref, _ = _oracle(ref, xs, np.zeros_like(y), np.zeros_like(gs), V, s)
    assert _rel(plan.residual(T(x[0]), None, None, T(V)), r0_ref) < 1e-10
    ga_ref, gg_ref = _ref_grads(ref, xs, y, gs, V, s)
    ga, gg = plan.residual_grad(T(x[0]), T(y), T(g[0]), T(V), T(s), want_grad_g=True)
    assert _rel(ga[None], ga_ref.sum(0)[None]) < 1e-10 and _rel(gg[None], gg_ref.sum(0)[None]) < 1e-10


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("mesh", MESHES, ids=["pixel", "cell"])
@pytest.mark.parametrize("m", [8, 40])
def test_identical_matrices_give_the_shared_results(m, mesh, dtype, dev):
    nx, ny, pixel = mesh
    plan, ref = _case(nx, ny, pixel, not pixel, dev)
    B = 6
    x, y, g, V, s = _inputs(plan, ref, B, m, "NDP", seed=m)
    T = lambda t: torch.tensor(t, dtype=dtype, device=dev)
    V2 = T(V[0])
    V3 = V2.expand(B, -1, -1).contiguous()
    tol = 1e-12 if dtype == torch.float64 else 1e-5   # FP32: the shared route keeps rho in FP64, this one as floats
    assert _rel(plan.residual(T(x), T(y), T(g), V3), plan.residual(T(x), T(y), T(g), V2).double().cpu().numpy()) < tol
    assert _rel(plan.residual_T(T(x), V3, T(s)), plan.residual_T(T(x), V2, T(s)).double().cpu().numpy()) < tol
    ga3, gg3 = plan.residual_grad(T(x), T(y), T(g), V3, T(s), want_grad_g=True)
    ga2, gg2 = plan.residual_grad(T(x), T(y), T(g), V2, T(s), want_grad_g=True)
    assert _rel(ga3, ga2.double().cpu().numpy()) < tol and _rel(gg3, gg2.double().cpu().numpy()) < tol


def test_gradcheck_through_the_autograd_function(dev):
    from gpde_b200.VirtualObservables import VoResidualFn
    plan, ref = _case(4, 3, False, False, dev)
    x, y, g, V, _ = _inputs(plan, ref, 2, 3, "NDP", seed=11)
    T = lambda t: torch.tensor(t, dtype=torch.float64, device=dev)
    V3 = T(V)
    fn = lambda yy, aa, gg: VoResidualFn.apply(yy, aa, gg, V3, plan, True)
    assert torch.autograd.gradcheck(fn, (T(y).requires_grad_(True), T(x).requires_grad_(True), T(g).requires_grad_(True)))


def _ensemble(dev, flux=False, N_gaussian=2, N_rbf=3):
    from conftest import load_golden
    from gpde_b200 import VirtualObservables as VO
    from gpde_b200.physics import setup_physics, BoundaryConditionEnsemble
    gold = load_golden("vo_2x2_8_nd")
    ph = setup_physics(int(gold['nx']), int(gold['nx']), int(gold['refines']), str(gold['kind']))
    bce = BoundaryConditionEnsemble(ph, gold['in_X_DG'].shape[0], str(gold['kind']), coefficients=gold['in_bc_coef'])
    qpe = VO.QuerryPointEnsemble.FromArrays(gold['in_X_DG'], bce, ph['fom'])
    np.random.seed(5)
    qe = VO.QuerryEnsemble.FromQuerryPointEnsemble(qpe, ph, CGR=True, flux=flux, N_gaussian=N_gaussian, N_rbf=N_rbf,
                                                   l_rbf=0.2, dtype=torch.double, device=dev)
    return VO.VirtualObservablesEnsemble(qpe, qe, torch.double, dev), qe, gold


def test_ensemble_residuals_with_per_sample_samplers(dev):
    ens, qe, gold = _ensemble(dev)
    Y = torch.tensor(gold['in_Y'], device=dev)
    N, m = Y.shape[0], qe[0].m
    assert qe[0].V is not qe[1].V
    r = ens.residuals(Y)
    S = torch.tensor(np.random.RandomState(1).standard_normal((N, m)), device=dev)
    q = ens.residual_gradients(S)
    for n in range(N):
        want_r = (qe[n].Gamma @ Y[n] - qe[n].alpha).cpu().numpy()
        assert _rel(r[n:n + 1], want_r[None]) < 1e-10
        want_q = (qe[n].GammaTransposed @ S[n]).cpu().numpy()
        assert _rel(q[n:n + 1], want_q[None]) < 1e-10
    # an explicit shared V behaves as before
    W = qe[0]._sampler._samplers[0]._W
    plan, a, G = ens._inputs()
    assert _rel(ens.residuals(Y, W), plan.residual(a, Y, G, W, a_is_log=False).cpu().numpy()) < 1e-13
    # only the project's kernels run (no cuBLAS / cuSOLVER)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ens.residuals(Y)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "Memcpy" not in e.name
             and "Memset" not in e.name]
    assert names and all("gpde" in n for n in names), names


def test_ensemble_without_weighting_matrices_raises(dev):
    ens, qe, gold = _ensemble(dev, flux=True, N_gaussian=0, N_rbf=0)
    assert qe[0].V is None
    Y = torch.tensor(gold['in_Y'], device=dev)
    with pytest.raises(RuntimeError, match="flux"):
        ens.residuals(Y)
    with pytest.raises(RuntimeError, match="flux"):
        ens.residual_gradients(torch.zeros(Y.shape[0], qe[0].m, dtype=torch.double, device=dev))


def test_empty_batch_in_either_layout(dev):
    plan, ref = _case(16, 8, True, False, dev)
    x, y, g, V, s = (torch.tensor(t, device=dev) for t in _inputs(plan, ref, 2, 5, "NDP", seed=2))
    assert plan.residual(x[:0], y[:0], g[:0], V[:0]).shape == (0, 5)
    assert plan.residual_T(x[:0], V[:0], s[:0]).shape == (0, plan.d)
    ga, _ = plan.residual_grad(x[:0], y[:0], g[:0], V[:0], s[:0])
    assert ga.shape == (0, plan.n_inputs)
    lib = plan._lib
    # B = 0 through the C ABI: no-op even with NULL operands, in either layout
    for v_stride in (plan.d * 5, 0):
        assert lib.gpde_vo_residual_f64(plan.handle, None, 0, 1, None, None, 0, None, v_stride, 5, None, None, None, 0, 0,
                                        None) == 0
        assert lib.gpde_vo_residual_T_f64(plan.handle, None, 0, 1, None, v_stride, 5, None, None, None, 0, None) == 0
        assert lib.gpde_vo_residual_grad_f64(plan.handle, None, 0, 1, None, None, 0, None, v_stride, 5, None, None, None,
                                             None, 0, None) == 0


def test_bad_arguments_through_v_stride(dev):
    from gpde_b200 import _lib
    plan, ref = _case(16, 8, True, False, dev)
    B, m = 3, 5
    x, y, g, V, s = (torch.tensor(t, device=dev) for t in _inputs(plan, ref, B, m, "NDP", seed=4))
    lib, P = plan._lib, lambda t: _lib.ptr(t, dev)
    r = torch.empty(B, m, dtype=torch.float64, device=dev)
    q = torch.empty(B, plan.d, dtype=torch.float64, device=dev)
    ga = torch.empty(B, plan.n_inputs, dtype=torch.float64, device=dev)
    ws = torch.empty(int(lib.gpde_vo_workspace_bytes(plan.handle, B, m)) + 64, dtype=torch.uint8, device=dev)
    wsp, mis = P(ws), ctypes.c_void_p(ws.data_ptr() + 8)
    st = _lib.stream_of(dev)
    res = lambda Vp, stride, w, rr=P(r), mm=m, fl=0: lib.gpde_vo_residual_f64(plan.handle, P(x), plan.n_inputs, 1, P(y), P(g),
                                                                              plan.n_bc, Vp, stride, mm, rr, None, w, fl, B, st)
    resT = lambda Vp, stride, w, qq=P(q): lib.gpde_vo_residual_T_f64(plan.handle, P(x), plan.n_inputs, 1, Vp, stride, m,
                                                                     P(s), qq, w, B, st)
    grad = lambda Vp, stride, w, gg=P(s): lib.gpde_vo_residual_grad_f64(plan.handle, P(x), plan.n_inputs, 1, P(y), P(g),
                                                                        plan.n_bc, Vp, stride, m, gg, P(ga), None, w, B, st)
    good = plan.d * m
    for call in (res, resT, grad):
        assert call(P(V), good, wsp) == 0
        assert call(P(V), good + 1, wsp) == GPDE_ERR_ARG       # v_stride neither 0 nor d*m
        assert call(P(V), 1, wsp) == GPDE_ERR_ARG
        assert call(P(V), -good, wsp) == GPDE_ERR_ARG
        assert call(P(V), good, mis) == GPDE_ERR_ARG           # misaligned workspace
        assert call(P(V), good, None) == GPDE_ERR_ARG          # no workspace
        assert call(None, good, wsp) == GPDE_ERR_ARG           # no V
    assert res(P(V), good, wsp, rr=None) == GPDE_ERR_ARG
    assert res(P(V), 0, wsp, mm=0) == GPDE_ERR_ARG
    assert res(P(V), good, wsp, mm=0) == GPDE_ERR_ARG          # m = 0 (rho only) takes no V
    assert res(P(V), good, wsp, fl=2) == GPDE_ERR_ARG          # packed weights are a shared-V layout
    assert resT(P(V), good, wsp, qq=None) == GPDE_ERR_ARG
    assert grad(P(V), good, wsp, gg=None) == GPDE_ERR_ARG
    torch.cuda.synchronize()
    # the Python layer: the batch and d of a 3-D V are checked, and packing is a shared-V concept
    with pytest.raises(ValueError):
        plan.residual(x, y, g, V[:2])
    with pytest.raises(ValueError):
        plan.residual(x, y, g, V[:, :-1])
    with pytest.raises(ValueError):
        plan.residual_T(x, V[:2], s)
    with pytest.raises(ValueError):
        plan.residual_grad(x, y, g, V[:, :-1], s)
    with pytest.raises(ValueError):
        plan.pack_weights(V, B)


def test_batches_that_wrap_the_grid_stride_loops(dev):
    """More (sample, panel) and (sample, row tile) jobs than CTAs launched; against torch on the same rho."""
    plan, ref = _case(4, 3, False, False, dev)
    B = 64 * torch.cuda.get_device_properties(dev).multi_processor_count + 37
    m = 3
    x, y, g, V, s = (torch.tensor(t, device=dev) for t in _inputs(plan, ref, B, m, "NDP", seed=9))
    r, rho = plan.residual(x, y, g, V, want_rho=True)
    assert _rel(r, torch.einsum("bi,bim->bm", rho, V).cpu().numpy()) < 1e-12
    q = plan.residual_T(x, V, s)
    w = torch.einsum("bim,bm->bi", V, s)
    assert _rel(q, plan.residual(x, w, None, None, ignore_load=True)[1].cpu().numpy()) < 1e-12


def test_repeated_calls_are_bitwise_identical(dev):
    for nx, ny, pixel in MESHES:
        plan, ref = _case(nx, ny, pixel, not pixel, dev)
        x, y, g, V, s = (torch.tensor(t, device=dev) for t in _inputs(plan, ref, 33, 100, "NDP", seed=1))
        outs = [(plan.residual(x, y, g, V), plan.residual_T(x, V, s), plan.residual_grad(x, y, g, V, s, want_grad_g=True))
                for _ in range(2)]
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
        assert torch.equal(outs[0][2][0], outs[1][2][0]) and torch.equal(outs[0][2][1], outs[1][2][1])


@pytest.mark.parametrize("B", [1, 5, 300])
@pytest.mark.parametrize("m", [1, 25, 32, 33, 100, 256])
@pytest.mark.parametrize("per_sample", [False, True], ids=["shared", "per_sample"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("mesh", MESHES, ids=["pixel", "cell"])
def test_one_workspace_query_covers_the_family(mesh, dtype, per_sample, m, B, dev):
    """gpde_vo_workspace_bytes(plan, B, m) is enough for residual, residual_T and residual_grad in either layout: each call
    gets exactly that many bytes at the start of a larger buffer, must leave the sentinel bytes behind them as they were,
    and must give what it gives with a generous workspace."""
    from gpde_b200 import _lib
    nx, ny, pixel = mesh
    plan, _ = _case(nx, ny, pixel, not pixel, dev)
    lib, P, st, sfx = plan._lib, (lambda t: _lib.ptr(t, dev)), _lib.stream_of(dev), _lib.suffix(dtype)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1000 * B + m)
    R = lambda *shape: torch.randn(*shape, generator=gen, device=dev, dtype=torch.float64).to(dtype)
    x, y, g, s = 0.6 * R(B, plan.n_inputs), R(B, plan.d), R(B, plan.n_bc), R(B, m)
    V = R(B, plan.d, m) if per_sample else R(plan.d, m)
    v_stride = plan.d * m if per_sample else 0
    need = int(lib.gpde_vo_workspace_bytes(plan.handle, B, m))

    def run(ws, after_each):
        r, q = (torch.empty(B, n, dtype=dtype, device=dev) for n in (m, plan.d))
        ga, gg = (torch.empty(B, n, dtype=dtype, device=dev) for n in (plan.n_inputs, plan.n_bc))
        calls = [lambda: getattr(lib, "gpde_vo_residual_" + sfx)(plan.handle, P(x), plan.n_inputs, 1, P(y), P(g), plan.n_bc,
                                                                 P(V), v_stride, m, P(r), None, P(ws), 0, B, st),
                 lambda: getattr(lib, "gpde_vo_residual_T_" + sfx)(plan.handle, P(x), plan.n_inputs, 1, P(V), v_stride, m,
                                                                   P(s), P(q), P(ws), B, st),
                 lambda: getattr(lib, "gpde_vo_residual_grad_" + sfx)(plan.handle, P(x), plan.n_inputs, 1, P(y), P(g),
                                                                      plan.n_bc, P(V), v_stride, m, P(s), P(ga), P(gg),
                                                                      P(ws), B, st)]
        for name, call in zip(("residual", "residual_T", "residual_grad"), calls):
            assert call() == 0, name
            after_each(name)
        return r, q, ga, gg

    buf = torch.full((need + (1 << 16),), 0xA5, dtype=torch.uint8, device=dev)

    def tail_intact(name):
        torch.cuda.synchronize()
        assert bool((buf[need:] == 0xA5).all()), "%s wrote past gpde_vo_workspace_bytes = %d" % (name, need)

    exact = run(buf[:need], tail_intact)
    generous = run(torch.empty(2 * need + (1 << 20), dtype=torch.uint8, device=dev), lambda name: None)
    for got, want in zip(exact, generous):
        assert torch.equal(got, want)

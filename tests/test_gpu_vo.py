"""GPU parity of the virtual-observable path (csrc/vo.cu through the C ABI and the VirtualObservables
mirrors) against the oracle and the reference-generated golden vectors (FP64 <= 1e-10, FP32 <= 1e-5)."""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def _setup(g, dev, kind=None):
    from gpde_b200.physics import setup_physics, BoundaryConditionEnsemble
    ph = setup_physics(int(g['nx']), int(g['nx']), int(g['refines']), str(g['kind']))
    N = g['in_X_DG'].shape[0]
    bce = BoundaryConditionEnsemble(ph, N, str(g['kind']), coefficients=g['in_bc_coef'])
    assert np.allclose(bce.constrained_dofs_values('fom'), g['in_g_fom'], atol=1e-15)
    return ph, bce


@pytest.mark.parametrize("name", ["vo_4x4_32_ndp", "vo_2x2_8_nd"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_residual_kernels_against_reference_vectors(name, dtype, dev):
    from gpde_b200.VirtualObservables import VoPlan
    g = load_golden(name)
    ph, bce = _setup(g, dev)
    plan = VoPlan.cached(ph['fom'], dev)
    a = torch.tensor(g['in_X_DG'], dtype=dtype, device=dev)
    y = torch.tensor(g['in_Y'], dtype=dtype, device=dev)
    gv = torch.tensor(g['in_g_fom'], dtype=dtype, device=dev)
    V = torch.tensor(g['in_V'], dtype=dtype, device=dev)
    r, rho = plan.residual(a, y, gv, V, want_rho=True)
    if dtype == torch.float64:
        want_r = g['out_residual']
        Gam, alp = g['out_Gamma'], g['out_alpha']
        tol = 1e-10
    else:   # oracle on the float32-rounded inputs
        from oracle import fem_p1, vo_ref
        P = fem_p1.build_problem(int(g['nx']), int(g['nx']), int(g['refines']))
        Vd = V.double().cpu().numpy()
        want_r, Gam, alp = [], [], []
        for n in range(a.shape[0]):
            K, f = fem_p1.assemble_system_free(P['coords_fom'], P['cells_fom'], np.exp(a[n].double().cpu().numpy()),
                                               P['bc_dofs_fom'], gv[n].double().cpu().numpy(), P['free_dofs_fom'])
            Ga, al = vo_ref.construct_querry_weak_galerkin(K, f, Vd)
            Gam.append(Ga); alp.append(al)
            want_r.append(Ga @ y[n].double().cpu().numpy() - al)
        want_r, Gam, alp = np.stack(want_r), np.stack(Gam), np.stack(alp)
        tol = 1e-5
    assert rel_err(r.cpu(), want_r) < tol
    # rho is the fine residual itself: r = rho V
    assert rel_err((rho.double() @ V.double()).cpu(), want_r) < (1e-10 if dtype == torch.float64 else 1e-5)
    # transposed application q = K_ff V s = Gamma^T s
    s = torch.tensor(np.random.RandomState(0).normal(size=(a.shape[0], V.shape[1])), dtype=dtype, device=dev)
    q = plan.residual_T(a, V, s)
    want_q = np.einsum('nmd,nm->nd', Gam, s.double().cpu().numpy())
    assert rel_err(q.cpu(), want_q) < tol
    # shared field (a_stride = 0) and shared Dirichlet data
    r0 = plan.residual(a[0], y, gv[0], V)
    r0_ref = np.stack([Gam[0] @ y[n].double().cpu().numpy() - alp[0] for n in range(a.shape[0])])
    assert rel_err(r0.cpu(), r0_ref) < tol


@pytest.mark.parametrize("name", ["vo_4x4_32_ndp", "vo_2x2_8_nd"])
def test_gamma_alpha_and_posterior_update_against_reference_vectors(name, dev):
    from gpde_b200 import VirtualObservables as VO
    g = load_golden(name)
    ph, bce = _setup(g, dev)
    V, mask = g['in_V'], g['in_mask']

    class FixedSampler(VO.BaseSampler):
        is_constant = True

        def __init__(self, qp):
            super().__init__(qp)
            self.m = V.shape[1]

        precision_mask = property(lambda self: mask)

        def _sample(self):
            return V

    qpe = VO.QuerryPointEnsemble.FromArrays(g['in_X_DG'], bce, ph['fom'], device=dev)
    qe = VO.QuerryEnsemble([VO.LinearQuerry(qp, FixedSampler(qp), torch.double, dev) for qp in qpe], torch.double, dev)
    for n, q in enumerate(qe):
        assert q.Gamma.dtype == torch.double and q.Gamma.shape == g['out_Gamma'][n].shape
        assert rel_err(q.Gamma.cpu(), g['out_Gamma'][n]) < 1e-12
        assert rel_err(q.alpha.cpu(), g['out_alpha'][n]) < 1e-11
        assert torch.equal(q.GammaTransposed, q.Gamma.t())
    Gn, an = qpe[0].construct_querry_weak_galerkin(V)          # numpy flavour of the reference API
    assert isinstance(Gn, np.ndarray) and rel_err(Gn, g['out_Gamma'][0]) < 1e-12 and rel_err(an, g['out_alpha'][0]) < 1e-11

    ens = VO.VirtualObservablesEnsemble(qpe, qe, torch.double, dev)
    assert ens.N == g['in_Y'].shape[0] and ens.m == V.shape[1] and ens.dim_out == g['in_Y'].shape[1]
    assert not ens.fixed_precision
    ens.update(torch.tensor(g['in_Y'], device=dev), torch.tensor(g['in_PREC1'], device=dev), 0)
    assert rel_err(ens.mean.cpu(), g['out_mean1']) < 1e-9
    assert rel_err(ens.vars.cpu(), g['out_vars1']) < 1e-8
    ens.update(torch.tensor(g['in_G2'], device=dev), torch.tensor(g['in_PREC2'], device=dev), 1)
    assert rel_err(ens._prec_beta.cpu(), g['out_prec_beta']) < 1e-8
    assert rel_err(ens._mean_vo_variances.cpu(), g['out_mean_vo_variances']) < 1e-8
    assert rel_err(ens.mean.cpu(), g['out_mean2']) < 1e-8
    assert rel_err(ens.vars.cpu(), g['out_vars2']) < 1e-7
    assert rel_err(ens.logsigma.cpu(), 0.5 * np.log(g['out_vars2'])) < 1e-7
    # single data point through VirtualObservable.update == the batched ensemble pass
    vo = ens[1]
    keep = vo.mean.clone()
    vo.update(torch.tensor(g['in_G2'][1], device=dev), torch.tensor(g['in_PREC2'][1], device=dev), 1, ForceUpdate=True)
    assert rel_err(vo.mean.cpu(), keep.cpu()) < 1e-12
    with pytest.raises(RuntimeError):
        vo.update(None, None, 0)
    # all residuals of the ensemble in one launch
    r = ens.residuals(torch.tensor(g['in_Y'], device=dev), V)
    assert rel_err(r.cpu(), g['out_residual']) < 1e-10
    # the ensemble keeps V packed between calls (same tensor, same version) and repacks after an in-place change
    assert torch.equal(ens.residuals(torch.tensor(g['in_Y'], device=dev), V), r)
    if torch.is_tensor(V) and V.dtype == torch.float64 and V.is_cuda:
        V.mul_(2.0)
        assert rel_err(ens.residuals(torch.tensor(g['in_Y'], device=dev), V).cpu(), 2.0 * g['out_residual']) < 1e-10
        V.mul_(0.5)


def test_reference_style_construction_and_samplers(dev):
    """QuerryEnsemble.FromQuerryPointEnsemble with CGR + Gaussian + RBF samplers, resample()."""
    from gpde_b200 import VirtualObservables as VO
    from oracle import fem_p1, vo_ref
    g = load_golden("vo_2x2_8_nd")
    ph, bce = _setup(g, dev)
    qpe = VO.QuerryPointEnsemble.FromArrays(g['in_X_DG'], bce, ph['fom'])
    np.random.seed(5)
    qe = VO.QuerryEnsemble.FromQuerryPointEnsemble(qpe, ph, CGR=True, flux=False, N_gaussian=2, N_rbf=3, l_rbf=0.2,
                                                   dtype=torch.double, device=dev)
    assert qe.N == len(qpe) and qe[0].m == ph['W'].shape[1] + 5 and qe.m == qe.N * qe[0].m
    assert np.all(qe.precision_mask < 0)
    ens = VO.VirtualObservablesEnsemble(qpe, qe, torch.double, dev)
    assert ens.fixed_precision
    P = fem_p1.build_problem(2, 2, 2)
    K, f = fem_p1.assemble_system_free(P['coords_fom'], P['cells_fom'], np.exp(g['in_X_DG'][0]), P['bc_dofs_fom'],
                                       g['in_g_fom'][0], P['free_dofs_fom'])
    # the CGR block of Gamma is W^T K
    Gam0, al0 = vo_ref.construct_querry_weak_galerkin(K, f, ph['W'])
    assert rel_err(qe[0].Gamma[:ph['W'].shape[1]].cpu(), Gam0) < 1e-12
    before = qe[0].Gamma.clone()
    ens.resample()
    after = qe[0].Gamma
    assert rel_err(after[:ph['W'].shape[1]].cpu(), Gam0) < 1e-12
    assert not torch.equal(before[-5:], after[-5:])               # random samplers were redrawn
    # infinite precision: the posterior mean satisfies Gamma mean = alpha
    N, d = g['in_Y'].shape
    ens.update(torch.tensor(g['in_Y'], device=dev), torch.full((N, d), 100.0, dtype=torch.double, device=dev), 0)
    for n in range(N):
        res = qe[n].Gamma @ ens.mean[n] - qe[n].alpha
        assert res.abs().max() < 1e-8
    # flux constraints (VirtualObservables.py:514-527): one learnable-precision row per coarse cell after the CGR block
    qe_flux = VO.QuerryEnsemble.FromQuerryPointEnsemble(qpe, ph, True, True, 0, 0, dtype=torch.double, device=dev)
    assert qe_flux[0].m == ph['W'].shape[1] + ph['rom'].mesh.num_cells and qe_flux[0].V is None


def test_pixel_input_plan_matches_cell_input_plan(dev):
    from gpde_b200.VirtualObservables import VoPlan
    from gpde_b200.workloads import Workload
    w = Workload("cfg1", B=7, seed=3)
    fom = w.physics['fom']
    pix_plan, cell_plan = VoPlan.cached(fom, dev, pixel_input=True), VoPlan.cached(fom, dev)
    img = torch.tensor(w.log_image, device=dev)
    X_DG = img[:, torch.tensor(fom.mesh.pixel_of_cell(), device=dev)]
    y, gv, V = (torch.tensor(t, device=dev) for t in (w.y, w.g_fom, w.V))
    # pixel input runs on the structured-grid kernel, cell input on the generic fused kernel
    assert pix_plan.kernel_path(V.shape[1]) == 2 and cell_plan.kernel_path(V.shape[1]) == 1
    assert rel_err(pix_plan.residual(img, y, gv, V).cpu(), cell_plan.residual(X_DG, y, gv, V).cpu()) < 1e-12
    assert pix_plan.n_inputs == 1024 and cell_plan.n_inputs == 2048 and pix_plan.slots_per_row == 6


def test_autograd_through_residual(dev):
    from gpde_b200.VirtualObservables import VoPlan, VoResidualFn
    from gpde_b200.workloads import Workload
    w = Workload("cfg1", B=2, seed=1)
    plan = VoPlan.cached(w.physics['fom'], dev, pixel_input=True)
    a, gv, V = (torch.tensor(t, device=dev) for t in (w.log_image, w.g_fom, w.V[:, :4].copy()))
    y = torch.tensor(w.y, device=dev, requires_grad=True)
    # 0.5 |r|^2 -> dL/dy = K_ff V r; compare with finite differences along a random direction
    r = VoResidualFn.apply(y, a, gv, V, plan, True)
    (0.5 * (r ** 2).sum()).backward()
    dirn = torch.randn_like(y)
    eps = 1e-6
    lp = 0.5 * (plan.residual(a, y.detach() + eps * dirn, gv, V) ** 2).sum()
    lm = 0.5 * (plan.residual(a, y.detach() - eps * dirn, gv, V) ** 2).sum()
    fd = (lp - lm) / (2 * eps)
    assert abs(fd.item() - (y.grad * dirn).sum().item()) < 1e-6 * max(1.0, abs(fd.item()))


@pytest.mark.parametrize("diag", ["right", "alternating"])
def test_other_fine_mesh_patterns(diag, dev):
    """The fine connectivity is an input of the plan (SURVEY.md section 7: refine() may give either)."""
    from gpde_b200.physics import setup_physics, BoundaryConditionEnsemble
    from gpde_b200.VirtualObservables import VoPlan
    from oracle import fem_p1, vo_ref
    ph = setup_physics(2, 2, 3, "NDP", diagonal=diag)
    rng = np.random.RandomState(2)
    bce = BoundaryConditionEnsemble(ph, 3, "NDP", rng=rng)
    fom = ph['fom']
    X = rng.normal(0.4, 0.8, size=(3, fom.dim_in))
    Y = rng.normal(size=(3, fom.dim_out))
    V = rng.normal(size=(fom.dim_out, 7))
    plan = VoPlan(fom, dev)
    r = plan.residual(torch.tensor(X, device=dev), torch.tensor(Y, device=dev),
                      torch.tensor(bce.constrained_dofs_values('fom'), device=dev), torch.tensor(V, device=dev))
    c, cells = fem_p1.unit_square_mesh(16, 16, diag)
    bc, _, free = fem_p1.dirichlet_left_right(c, 'ND')
    for n in range(3):
        K, f = fem_p1.assemble_system_free(c, cells, np.exp(X[n]), bc, bce.constrained_dofs_values('fom')[n], free)
        assert rel_err(r[n].cpu(), vo_ref.vo_residual(K, f, V, Y[n])) < 1e-10
    assert plan.slots_per_row == (6 if diag == "right" else 8)


def test_full_size_properties_config2(dev):
    """64x64 FOM, batch 4096 (BASELINE config 2): closed-form zero residual, linearity, r = rho V."""
    from gpde_b200.VirtualObservables import VoPlan
    from gpde_b200.workloads import Workload
    w = Workload("cfg2", B=4096, seed=0)
    fom = w.physics['fom']
    plan = VoPlan.cached(fom, dev, pixel_input=True)
    V = torch.tensor(w.V, device=dev)
    gv = torch.tensor(w.g_fom[0], device=dev)            # ND: shared Dirichlet data
    B = w.B
    gen = torch.Generator().manual_seed(1)
    # uniform medium (a different constant per sample): y = x-coordinate solves the PDE exactly
    a_u = torch.randn(B, 1, generator=gen, dtype=torch.float64).expand(B, w.P).contiguous().to(dev)
    yx = torch.tensor(fom.mesh.coords[fom.free_dofs, 0], device=dev).expand(B, -1).contiguous()
    r, rho = plan.residual(a_u, yx, gv, V, want_rho=True)
    assert rho.abs().max() < 1e-11 and r.abs().max() < 1e-11
    # linearity in (y, g): r(y1 + y2, 2g) - r(y1, g) - r(y2, g) = 0, random log-normal fields
    a = torch.tensor(w.log_image, device=dev)
    y1 = torch.tensor(w.y, device=dev)
    y2 = torch.randn(B, w.d, generator=gen, dtype=torch.float64).to(dev)
    r1, r2, r12 = plan.residual(a, y1, gv, V), plan.residual(a, y2, gv, V), plan.residual(a, y1 + y2, 2 * gv, V)
    assert rel_err((r1 + r2).cpu(), r12.cpu()) < 1e-12
    # sample independence (bitwise) and r = rho V
    perm = torch.randperm(B, generator=gen).to(dev)
    assert torch.equal(plan.residual(a[perm], y1[perm], gv, V), r1[perm])
    _, rho1 = plan.residual(a, y1, gv, V, want_rho=True)
    assert rel_err((rho1 @ V).cpu(), r1.cpu()) < 1e-12
    # transposed op is the adjoint of the residual map: <s, Gamma y> = <Gamma^T s, y>  (g = 0, no load)
    s = torch.randn(B, w.m, generator=gen, dtype=torch.float64).to(dev)
    lhs = (s * plan.residual(a, y2, None, V, ignore_load=True)).sum(dim=1)
    rhs = (plan.residual_T(a, V, s) * y2).sum(dim=1)
    assert rel_err(lhs.cpu(), rhs.cpu()) < 1e-11


def test_schedules_and_guards(dev):
    from gpde_b200 import VirtualObservables as VO, _lib
    lin = VO.LinearTemperatureSchedule(1.0, 1e-4, 11)
    assert lin.get_temperature(0) == 1.0 and abs(lin.get_temperature(10) - 1e-4) < 1e-15
    ex = VO.ExponentialTemperatureSchedule(1.0, 1e-4, 11)
    assert abs(ex.get_temperature(5) - 1e-2) < 1e-12
    with pytest.raises(RuntimeError):
        lin.get_temperature(12)
    from gpde_b200.physics import setup_physics
    ph = setup_physics(2, 2, 1)
    with pytest.raises(_lib.GpdeLibraryError):        # no CPU fallback
        VO.VoPlan(ph['fom'], torch.device("cpu"))


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_fused_path_matches_unfused_kernels(dtype, dev, monkeypatch):
    """The fused (edge form + ring staging + FP64 MMA) kernel against the version-1 kernels, including a
    ragged batch (B % 8 != 0), every column-tile variant (m <= 8, 16, 32) and m > 32 (unfused only)."""
    from gpde_b200.VirtualObservables import VoPlan
    from gpde_b200.workloads import Workload
    w = Workload("cfg1", B=21, seed=5)
    plan = VoPlan.cached(w.physics['fom'], dev, pixel_input=True)
    assert plan.fused_smem_bytes > 0
    # the experiment switches are read once, at plan creation: one plan per kernel family
    plan_fused, plan_v1 = plan.variant(GPDE_VO_PATH="fused"), plan.variant(GPDE_VO_PATH="v1")
    plan_fused_sync = plan.variant(GPDE_VO_PATH="fused", GPDE_VO_SYNC_STAGING="1")
    a, y, gv = (torch.tensor(t, dtype=dtype, device=dev) for t in (w.log_image, w.y, w.g_fom))
    rng = np.random.RandomState(0)
    tol = 1e-12 if dtype == torch.float64 else 2e-6
    for m in (1, 7, 8, 13, 16, 25, 32, 40):
        V = torch.tensor(rng.normal(size=(w.d, m)), dtype=dtype, device=dev)
        s = torch.tensor(rng.normal(size=(21, m)), dtype=dtype, device=dev)
        assert plan_fused.kernel_path(m, dtype) == (1 if m <= 32 else 0)
        r2, rho2 = plan_fused.residual(a, y, gv, V, want_rho=True)
        q2 = plan_fused.residual_T(a, V, s)
        if m <= 32:
            assert rel_err(plan_fused.residual(a, y, gv, V).cpu(), r2.cpu()) == 0.0    # rho output does not change r
        assert plan_v1.launches_per_residual(m) == 3 and plan_v1.kernel_path(m, dtype) == 0
        r1, rho1 = plan_v1.residual(a, y, gv, V, want_rho=True)
        q1 = plan_v1.residual_T(a, V, s)
        assert rel_err(r2.cpu(), r1.cpu()) < tol, m
        assert rel_err(rho2.cpu(), rho1.cpu()) < tol, m
        assert rel_err(q2.cpu(), q1.cpu()) < tol, m
    # rho only (no weighting matrix)
    _, rho = plan.residual(a, y, gv, None)
    assert rel_err(rho.cpu(), rho1.cpu()) < tol
    # synchronous staging flavour of the fused kernel (what FP32 inputs and non-monotone rings use)
    V = torch.tensor(rng.normal(size=(w.d, 25)), dtype=dtype, device=dev)
    r3 = plan_fused_sync.residual(a, y, gv, V)
    assert torch.equal(r3, plan_fused.residual(a, y, gv, V))


def _grid_case(nx, ny, ptype, B, seed, dev, load=False):
    """Pixel-input plan on an nx x ny fine grid with random fields / data."""
    from gpde_b200 import fem
    from gpde_b200.physics import LinearEllipticPhysics, BoundaryConditionEnsemble
    from gpde_b200.VirtualObservables import VoPlan
    rng = np.random.RandomState(seed)
    mesh = fem.P1Mesh(nx, ny, "right")
    fom = LinearEllipticPhysics("fom", ptype, mesh)
    f = rng.normal(size=mesh.num_nodes) if load else None
    plan = VoPlan(fom, dev, mesh.pixel_of_cell(), nx * ny, load=f)
    bc = mesh.dirichlet_dofs()[0]
    g = rng.uniform(-0.5, 0.5, size=(B, bc.size))
    a = rng.normal(0.4, 0.8, size=(B, nx * ny))
    y = rng.normal(size=(B, fom.dim_out))
    return plan, fom, a, y, g, rng


@pytest.mark.parametrize("nx,ny,B", [(64, 64, 37), (32, 32, 64), (8, 8, 3), (2, 1, 5), (4, 7, 9), (18, 5, 33),
                                     (34, 3, 8), (66, 2, 17), (128, 16, 19), (130, 4, 16), (200, 3, 9)])
def test_pixel_plans_with_a_load_match_generic_kernels(nx, ny, B, dev, monkeypatch):
    """Pixel-input plans with a load vector against the generic kernels on the same inputs: widths that are / are not
    multiples of 16, tiny grids, ragged batches, every column-tile variant, odd batch x odd d (y ends off a 16-byte
    boundary), shared field / Dirichlet data, conductivity (not log) input, load vector on / off.  The lean grid kernel
    does not subtract a load: these calls take the generic kernels unless they ignore it."""
    load = True
    plan, fom, a, y, g, rng = _grid_case(nx, ny, "NDP", B, nx * 1000 + ny, dev, load=load)
    plan_v1 = plan.variant(GPDE_VO_PATH="v1")
    T = lambda t: torch.tensor(t, device=dev)
    lean = nx in (16, 32, 64, 128) and ny % 2 == 0 and not load
    for m in (1, 8, 9, 16, 25, 32, 33, 70, 130):
        V = T(rng.normal(size=(fom.dim_out, m)))
        path = (2 if m <= 32 else 3) if lean else (1 if m <= 32 and plan.fused_smem_bytes > 0 else 0)
        assert plan.kernel_path(m) == path and plan.launches_per_residual(m) == {3: 3, 2: 2, 1: 1, 0: 3}[path]
        assert plan.kernel_path(m, torch.float64) == plan.kernel_path(m, torch.float32)
        variants = [
            dict(a=T(a), y=T(y), g=T(g)),
            dict(a=T(a[0]), y=T(y), g=T(g[0])),                  # shared field and Dirichlet data
            dict(a=T(np.exp(a)), y=T(y), g=None, a_is_log=False),
            dict(a=T(a), y=T(y), g=T(g), ignore_load=True),
        ]
        for kw in variants:
            aa, yy, gg = kw.pop('a'), kw.pop('y'), kw.pop('g')
            r_grid = plan.residual(aa, yy, gg, V, **kw)
            r_v1 = plan_v1.residual(aa, yy, gg, V, **kw)
            assert rel_err(r_grid.cpu(), r_v1.cpu()) < 1e-12, (m, sorted(kw))
    # transposed application q = K_ff (V s): tensor-core expansion + marching kernel against the generic kernels
    for m in (1, 25, 70):
        V = T(rng.normal(size=(fom.dim_out, m)))
        sv = T(rng.normal(size=(B, m)))
        for kw in (dict(a=T(a)), dict(a=T(a[0])), dict(a=T(np.exp(a)), a_is_log=False)):
            aa = kw.pop('a')
            q_grid = plan.residual_T(aa, V, sv, **kw)
            q_v1 = plan_v1.residual_T(aa, V, sv, **kw)
            assert rel_err(q_grid.cpu(), q_v1.cpu()) < 1e-12, (m, sorted(kw))
    # unaligned views (odd storage offsets) are served by the generic kernels, same numbers
    V = T(rng.normal(size=(fom.dim_out, 25)))
    big = torch.zeros(B * fom.dim_out + 1, dtype=torch.float64, device=dev)
    yv = big[1:].view(B, fom.dim_out)
    yv.copy_(T(y))
    assert rel_err(plan.residual(T(a), yv, T(g), V).cpu(), plan.residual(T(a), T(y), T(g), V).cpu()) < 1e-12


@pytest.mark.parametrize("nx,ny,B", [(64, 64, 37), (32, 32, 64), (16, 2, 130), (16, 6, 3), (128, 4, 19), (64, 2, 1),
                                     (32, 8, 129)])
def test_lean_grid_kernel_matches_generic_kernels(nx, ny, B, dev, monkeypatch):
    """vo_grid2.cuh (nx in {16,32,64,128}, even ny, no load) against the version-1 kernels: every (n-tiles, DFMA column)
    split of m, ragged batches (incl. batches smaller than a CTA), y views starting off a 16-byte boundary (both phases),
    shared field / Dirichlet rows, no Dirichlet data, conductivity input, the rho variant behind residual_T and m > 32."""
    plan, fom, a, y, g, rng = _grid_case(nx, ny, "NDP", B, nx * 77 + ny, dev, load=False)
    plan_v1 = plan.variant(GPDE_VO_PATH="v1")
    T = lambda t: torch.tensor(t, device=dev)
    big = torch.zeros(B * fom.dim_out + 1, dtype=torch.float64, device=dev)
    y_odd = big[1:].view(B, fom.dim_out)
    y_odd.copy_(T(y))
    for m in (1, 8, 9, 16, 17, 24, 25, 32, 40):
        V = T(rng.normal(size=(fom.dim_out, m)))
        variants = [
            dict(a=T(a), y=T(y), g=T(g)),
            dict(a=T(a), y=y_odd, g=T(g)),
            dict(a=T(a[0]), y=T(y), g=T(g[0])),
            dict(a=T(np.exp(a)), y=T(y), g=None, a_is_log=False),
        ]
        for kw in variants:
            aa, yy, gg = kw.pop('a'), kw.pop('y'), kw.pop('g')
            r_lean = plan.residual(aa, yy, gg, V, **kw)
            r_v1 = plan_v1.residual(aa, yy, gg, V, **kw)
            assert rel_err(r_lean.cpu(), r_v1.cpu()) < 1e-12, (m, sorted(kw))
    for m in (1, 5, 8, 9, 16, 25, 28, 29, 32, 40):   # every k-step count of the expansion kernel (vo_expand.cuh), and m > 32
        V = T(rng.normal(size=(fom.dim_out, m)))
        sv = T(rng.normal(size=(B, m)))
        q_lean = plan.residual_T(T(a), V, sv)
        q_v1 = plan_v1.residual_T(T(a), V, sv)
        assert rel_err(q_lean.cpu(), q_v1.cpu()) < 1e-12, m
    # extreme log-conductivities take the libm exp() branch: same numbers as the generic kernels
    a2 = a.copy()
    a2[:, ::7] = -705.0
    a2[:, 3::11] = -750.0
    V = T(rng.normal(size=(fom.dim_out, 25)))
    r_lean = plan.residual(T(a2), T(y), T(g), V)
    r_v1 = plan_v1.residual(T(a2), T(y), T(g), V)
    assert torch.isfinite(r_v1).all() and rel_err(r_lean.cpu(), r_v1.cpu()) < 1e-12


@pytest.mark.parametrize("nx,ny,B", [(64, 64, 37), (32, 32, 64), (16, 2, 130), (16, 6, 3), (128, 4, 19), (64, 2, 1),
                                     (32, 8, 129)])
def test_lean_grid_kernel_fp32_io(nx, ny, B, dev):
    """FP32 I/O through the lean grid kernel (rows staged as floats, FP64 arithmetic): against the FP64 kernel on the
    float-rounded inputs, to output rounding.  Every n-tile split of m, ragged batches, y views at all four 4-byte phases
    of a 16-byte boundary (the last one ending exactly at the end of its allocation: tail copies), shared field /
    Dirichlet rows, conductivity input, the rho-only output, m > 32, residual_T and packed weights."""
    from gpde_b200.VirtualObservables import PackedWeights
    plan, fom, a, y, g, rng = _grid_case(nx, ny, "NDP", B, nx * 31 + ny, dev, load=False)
    d = fom.dim_out
    F = lambda t: torch.tensor(t, device=dev, dtype=torch.float32)
    D = lambda t: t.double()
    a32, y32, g32 = F(a), F(y), F(g)
    assert plan.kernel_path(25, torch.float32) == 2 and plan.kernel_path(40, torch.float32) == 3
    y_views = [y32]
    for off in (1, 2, 3):
        big = torch.zeros(B * d + off, dtype=torch.float32, device=dev)    # the view ends where the allocation ends
        v = big[off:].view(B, d)
        v.copy_(y32)
        y_views.append(v)
    tol = 2e-6
    for m in (1, 8, 9, 16, 17, 24, 25, 32):
        V32 = F(rng.normal(size=(d, m)))
        r_ref = plan.residual(D(a32), D(y32), D(g32), D(V32)).cpu()
        for yy in y_views:
            assert rel_err(plan.residual(a32, yy, g32, V32).double().cpu(), r_ref) < tol, m
        r_sh = plan.residual(a32[0], y32, g32[0], V32).double().cpu()
        assert rel_err(r_sh, plan.residual(D(a32[0]), D(y32), D(g32[0]), D(V32)).cpu()) < tol, m
        ea = torch.exp(D(a32)).float()
        r_lin = plan.residual(ea, y32, None, V32, a_is_log=False).double().cpu()
        assert rel_err(r_lin, plan.residual(D(ea), D(y32), None, D(V32), a_is_log=False).cpu()) < tol, m
    V32 = F(rng.normal(size=(d, 25)))
    pw = plan.pack_weights(V32, B)
    assert isinstance(pw, PackedWeights)
    assert torch.equal(plan.residual(a32, y32, g32, pw), plan.residual(a32, y32, g32, V32))
    _, rho32 = plan.residual(a32, y32, g32, None)                                   # the fine residual alone
    _, rho64 = plan.residual(D(a32), D(y32), D(g32), None)
    _, rho_v1 = plan.variant(GPDE_VO_PATH="v1").residual(D(a32), D(y32), D(g32), None)
    assert rel_err(rho64.cpu(), rho_v1.cpu()) < 1e-12
    assert rho32.dtype == torch.float32 and rel_err(rho32.double().cpu(), rho64.cpu()) < tol
    V40 = F(rng.normal(size=(d, 40)))                                                # rho kernel + FP64 contraction
    assert rel_err(plan.residual(a32, y32, g32, V40).double().cpu(), plan.residual(D(a32), D(y32), D(g32), D(V40)).cpu()) < tol
    for m in (5, 16, 25, 32):
        Vm, sv = F(rng.normal(size=(d, m))), F(rng.normal(size=(B, m)))
        q32 = plan.residual_T(a32, Vm, sv)
        assert q32.dtype == torch.float32
        assert rel_err(q32.double().cpu(), plan.residual_T(D(a32), D(Vm), D(sv)).cpu()) < tol, m


def test_packed_weights_give_the_same_residual(dev):
    """gpde_vo_pack_weights_f64 + flags bit1: V packed once, many residual calls; bitwise equal to the call that packs
    V itself; meshes without a packed layout hand the matrix back."""
    from gpde_b200.VirtualObservables import PackedWeights
    plan, fom, a, y, g, rng = _grid_case(32, 8, "NDP", 21, 5, dev, load=False)
    T = lambda t: torch.tensor(t, device=dev)
    for m in (7, 25, 32):
        V = T(rng.normal(size=(fom.dim_out, m)))
        pw = plan.pack_weights(V, 21)
        assert isinstance(pw, PackedWeights)
        r0 = plan.residual(T(a), T(y), T(g), V)
        for _ in range(2):
            assert torch.equal(plan.residual(T(a), T(y), T(g), pw), r0)
        assert torch.equal(plan.residual(T(a[:5]), T(y[:5]), T(g[:5]), pw), r0[:5])          # smaller batch
        r1, rho1 = plan.residual(T(a), T(y), T(g), pw, want_rho=True)                         # not a packed call: plain V
        assert rel_err(r1.cpu(), r0.cpu()) < 1e-12 and rel_err((rho1 @ V).cpu(), r0.cpu()) < 1e-12
        pw2 = plan.pack_weights(2.0 * V, 21, out=pw)                                          # buffer reuse
        assert pw2.buf.data_ptr() == pw.buf.data_ptr()
        assert rel_err(plan.residual(T(a), T(y), T(g), pw2).cpu(), 2.0 * r0.cpu()) < 1e-13
    assert torch.is_tensor(plan.pack_weights(T(rng.normal(size=(fom.dim_out, 40))), 21))      # m > 32
    plan2, fom2, a2, y2, g2, _ = _grid_case(18, 5, "NDP", 4, 6, dev, load=False)              # not a lean-kernel mesh
    V2 = T(rng.normal(size=(fom2.dim_out, 25)))
    assert torch.is_tensor(plan2.pack_weights(V2, 4))


def test_lean_grid_kernel_against_oracle(dev):
    """Lean grid kernel against the CPU oracle (restated FEniCS assembly + reference VO arithmetic), 1e-10."""
    from oracle import fem_p1, vo_ref
    nx, ny, B = 32, 10, 11
    plan, fom, a, y, g, rng = _grid_case(nx, ny, "NDP", B, 7, dev)
    V = rng.normal(size=(fom.dim_out, 25))
    assert plan.kernel_path(25) == 2
    r = plan.residual(torch.tensor(a, device=dev), torch.tensor(y, device=dev), torch.tensor(g, device=dev),
                      torch.tensor(V, device=dev)).cpu().numpy()
    c, cells = fem_p1.unit_square_mesh(nx, ny, "right")
    bc, _, free = fem_p1.dirichlet_left_right(c, 'ND')
    pix = fom.mesh.pixel_of_cell()
    for n in range(B):
        K, f = fem_p1.assemble_system_free(c, cells, np.exp(a[n][pix]), bc, g[n], free)
        assert rel_err(r[n], vo_ref.vo_residual(K, f, V, y[n])) < 1e-10


def test_unfused_kernels_against_reference_vectors(dev, monkeypatch):
    from gpde_b200.VirtualObservables import VoPlan
    g = load_golden("vo_4x4_32_ndp")
    ph, bce = _setup(g, dev)
    plan_v1 = VoPlan(ph['fom'], dev, experiment=dict(GPDE_VO_PATH="v1"))
    assert plan_v1.kernel_path(g['in_V'].shape[1]) == 0
    a, y, gv, V = (torch.tensor(g[k], device=dev) for k in ('in_X_DG', 'in_Y', 'in_g_fom', 'in_V'))
    assert rel_err(plan_v1.residual(a, y, gv, V).cpu(), g['out_residual']) < 1e-10


def test_full_size_properties_config3(dev, monkeypatch):
    """128x128 FOM with 256 weighting functions (BASELINE config 3 mesh and m; a 384-sample slice of the batch so the
    test stays short): grid rho kernel + FP64 tensor-core contraction against closed forms and the generic kernels."""
    from gpde_b200.VirtualObservables import VoPlan
    from gpde_b200.workloads import Workload
    w = Workload("cfg3", B=384, seed=0)
    fom = w.physics['fom']
    plan = VoPlan.cached(fom, dev, pixel_input=True)
    assert w.m == 256 and w.d == 16383 and plan.kernel_path(w.m) == 3 and plan.launches_per_residual(w.m) == 3
    plan_v1 = plan.variant(GPDE_VO_PATH="v1")
    V = torch.tensor(w.V, device=dev)
    gv = torch.tensor(w.g_fom[0], device=dev)
    B = w.B
    gen = torch.Generator().manual_seed(3)
    # uniform medium: y = x solves the PDE exactly -> r = 0 (relative to the size of the terms that cancel)
    a_u = torch.randn(B, 1, generator=gen, dtype=torch.float64).expand(B, w.P).contiguous().to(dev)
    yx = torch.tensor(fom.mesh.coords[fom.free_dofs, 0], device=dev).expand(B, -1).contiguous()
    assert plan.residual(a_u, yx, gv, V).abs().max() < 1e-10
    a = torch.tensor(w.log_image, device=dev)
    y1 = torch.tensor(w.y, device=dev)
    y2 = torch.randn(B, w.d, generator=gen, dtype=torch.float64).to(dev)
    r1 = plan.residual(a, y1, gv, V)
    # against the generic kernels (matvec + the same contraction) on the same inputs
    r1_v1, rho_v1 = plan_v1.residual(a, y1, gv, V, want_rho=True)
    assert rel_err(r1.cpu(), r1_v1.cpu()) < 1e-12
    assert rel_err((rho_v1 @ V).cpu(), r1.cpu()) < 1e-12       # torch / cuBLAS FP64 as a third opinion
    # linearity, ragged tail (B % 128 != 0 for the 128-row GEMM tiles), sample independence
    r2, r12 = plan.residual(a, y2, gv, V), plan.residual(a, y1 + y2, 2 * gv, V)
    assert rel_err((r1 + r2).cpu(), r12.cpu()) < 1e-12
    assert torch.equal(plan.residual(a[:131], y1[:131], gv, V), r1[:131])
    # adjointness with the transposed application
    s = torch.randn(B, w.m, generator=gen, dtype=torch.float64).to(dev)
    lhs = (s * plan.residual(a, y2, None, V, ignore_load=True)).sum(dim=1)
    rhs = (plan.residual_T(a, V, s) * y2).sum(dim=1)
    assert rel_err(lhs.cpu(), rhs.cpu()) < 1e-11


def test_empty_batch_and_single_sample(dev):
    plan, fom, a, y, g, rng = _grid_case(16, 16, "NDP", 3, 11, dev)
    T = lambda t: torch.tensor(t, device=dev)
    V = T(rng.normal(size=(fom.dim_out, 25)))
    r = plan.residual(T(a[:0]), T(y[:0]), T(g[:0]), V)
    assert r.shape == (0, 25)
    r1 = plan.residual(T(a[:1]), T(y[:1]), T(g[:1]), V)
    assert rel_err(r1.cpu(), plan.residual(T(a), T(y), T(g), V)[:1].cpu()) == 0.0


def test_energy_virtual_observables_against_reference_vectors(dev):
    """EnergyVirtualObservablesEnsemble mirror (matrix-free subspace Newton on the device) against the reference's
    own output (tests/golden/energy_2x2_16_ndp.npz): temperature schedule, posterior mean and variances."""
    from gpde_b200 import VirtualObservables as VO
    g = load_golden("energy_2x2_16_ndp")
    ph, bce = _setup(g, dev)
    fom = ph['fom']
    N, n_it = g['in_X_DG'].shape[0], int(g['n_it'])
    qpe = VO.QuerryPointEnsemble.FromArrays(g['in_X_DG'], bce, fom, device=dev)

    class SequenceSampler(VO.BaseSampler):
        calls = 0

        def _sample(self):
            V = g['in_V_seq'][SequenceSampler.calls]
            SequenceSampler.calls += 1
            return V

    ens = VO.EnergyVirtualObservablesEnsemble(qpe, n_it, SequenceSampler(qpe[0]), torch.double, dev)
    ens.set_linear_temperature_schedule(T_init=1.0, T_final=1e-2, num_steps=4)
    with pytest.raises(RuntimeError):
        ens[0].update(torch.zeros(fom.dim_out), torch.ones(fom.dim_out), 0)          # ForceUpdate is mandatory (:772)
    for it in range(g['in_G'].shape[0]):
        ens.update(torch.tensor(g['in_G'][it], device=dev), torch.tensor(g['in_PREC'][it], device=dev), it)
        assert abs(ens[0].temperature - float(g['out_temperature'][it])) < 1e-15
        assert rel_err(ens.mean.cpu(), g['out_mean'][it]) < 1e-10
        assert rel_err(ens.vars.cpu(), g['out_vars'][it]) < 1e-12
        assert ens.logsigma.shape == (N, fom.dim_out) and ens.m == 1
    assert SequenceSampler.calls == g['in_V_seq'].shape[0]


def test_flux_constrain_sampler_wraps_a_setup_time_object(dev):
    """FluxConstrainSampler (VirtualObservables.py:323-349) takes (Gamma, alpha) from a flux-balance object built at
    setup; the mirror passes them through as float64 device tensors and concatenates with other samplers' masks."""
    from gpde_b200 import VirtualObservables as VO
    plan, fom, a, y, g, rng = _grid_case(8, 8, "NDP", 2, 5, dev)
    from gpde_b200.physics import BoundaryConditionEnsemble
    bce = BoundaryConditionEnsemble({'fom': fom, 'rom': fom}, 2, "NDP", rng=rng)
    qp = VO.QuerryPoint(fom, rng.normal(size=fom.dim_in), bce[0], device=dev)

    class FakeFlux(object):
        initialized = True

        def assemble_reduced(self, x, bc):
            assert np.all(x > 0)
            return rng.normal(size=(3, fom.dim_out)), rng.normal(size=3)

    s = VO.FluxConstrainSampler(qp, FakeFlux())
    Gam, alp = s.sample()
    assert s.m == 3 and s.is_constant and np.all(s.precision_mask == 1) and not s.fixed_precision
    assert Gam.dtype == torch.double and Gam.device.type == "cuda" and Gam.shape == (3, fom.dim_out) and alp.shape == (3,)
    FakeFlux.initialized = False
    with pytest.raises(RuntimeError):
        VO.FluxConstrainSampler(qp, FakeFlux())


def test_rbf_sampler_on_device_matches_host_evaluation(dev):
    """RadialBasisFunctionSampler: centres from numpy's stream in the reference's order, evaluation on the device
    (query points that live on a CUDA device) against the host evaluation (query points without a device)."""
    from gpde_b200 import VirtualObservables as VO
    g = load_golden("vo_2x2_8_nd")
    ph, bce = _setup(g, dev)
    qp_dev = VO.QuerryPoint(ph['fom'], g['in_X_DG'][0], bce[0], device=dev)
    qp_host = VO.QuerryPoint(ph['fom'], g['in_X_DG'][0], bce[0])
    np.random.seed(11)
    V_dev = VO.RadialBasisFunctionSampler(qp_dev, 0.2, 4).sample_V()
    np.random.seed(11)
    V_host = VO.RadialBasisFunctionSampler(qp_host, 0.2, 4).sample_V()
    assert isinstance(V_dev, torch.Tensor) and V_dev.device.type == "cuda" and isinstance(V_host, np.ndarray)
    assert rel_err(V_dev.cpu(), V_host) < 1e-14
    # concatenation with a host-side sampler ends up on the device
    np.random.seed(3)
    cat = VO.ConcatenatedSamplers([VO.GaussianSketchingSampler(qp_dev, 2), VO.RadialBasisFunctionSampler(qp_dev, 0.2, 3)])
    Vc = cat.sample_V()
    assert isinstance(Vc, torch.Tensor) and Vc.shape == (ph['fom'].dim_out, 5) and cat.m == 5
    Gam, alp = cat.sample()
    assert Gam.shape == (5, ph['fom'].dim_out) and alp.shape == (5,)


def test_gaussian_sketch_on_device(dev):
    """GaussianSketchingSampler (VirtualObservables.py:230-258): query points on a CUDA device draw the i.i.d. N(0,1)
    weighting vectors on the device; np.random.seed() still fixes the sequence; host query points keep the reference's
    numpy stream draw for draw."""
    from gpde_b200 import VirtualObservables as VO
    g = load_golden("vo_2x2_8_nd")
    ph, bce = _setup(g, dev)
    qp_dev = VO.QuerryPoint(ph['fom'], g['in_X_DG'][0], bce[0], device=dev)
    qp_host = VO.QuerryPoint(ph['fom'], g['in_X_DG'][0], bce[0])
    d = ph['fom'].dim_out
    np.random.seed(5)
    V1 = VO.GaussianSketchingSampler(qp_dev, 64).sample_V()
    V1b = VO.GaussianSketchingSampler(qp_dev, 64).sample_V()
    np.random.seed(5)
    V2 = VO.GaussianSketchingSampler(qp_dev, 64).sample_V()
    assert isinstance(V1, torch.Tensor) and V1.is_cuda and V1.dtype == torch.double and V1.shape == (d, 64)
    assert torch.equal(V1, V2) and not torch.equal(V1, V1b)
    assert abs(float(V1.mean())) < 0.1 and abs(float(V1.std()) - 1.0) < 0.1
    np.random.seed(5)
    Vh = VO.GaussianSketchingSampler(qp_host, 3).sample_V()
    np.random.seed(5)
    ref = np.stack([np.random.normal(0, 1, d) for _ in range(3)], axis=1)      # the reference's loop, :243-246
    assert isinstance(Vh, np.ndarray) and np.array_equal(Vh, ref)
    s = VO.GaussianSketchingSampler(qp_dev, 4)
    Gam, alp = s.sample()
    assert Gam.shape == (4, d) and alp.shape == (4,) and s.fixed_precision


@pytest.mark.parametrize("splits", [2, 4, 8])
def test_split_contraction_matches_single_pass(splits, dev):
    """m > 32: the FP64 tensor-core contraction cut into parts of the contraction length (tail of the tile grid on the SMs,
    vo_gemm.cuh) with the deterministic in-order reduction == the single-pass contraction to rounding; ragged batch; FP32
    I/O; repeated calls give bitwise the same numbers."""
    plan, fom, a, y, g, rng = _grid_case(64, 16, "NDP", 150, 21, dev, load=False)
    one, cut = plan.variant(GPDE_GEMM_SPLITS="1"), plan.variant(GPDE_GEMM_SPLITS=str(splits))
    T = lambda t: torch.tensor(t, device=dev)
    for m in (40, 100, 256):
        V = T(rng.normal(size=(fom.dim_out, m)))
        r1 = one.residual(T(a), T(y), T(g), V)
        r2 = cut.residual(T(a), T(y), T(g), V)
        assert rel_err(r2.cpu(), r1.cpu()) < 1e-13, m
        assert torch.equal(r2, cut.residual(T(a), T(y), T(g), V))
        r3 = cut.residual(T(a).float(), T(y).float(), T(g).float(), V.float())
        assert r3.dtype == torch.float32 and rel_err(r3.double().cpu(), r1.cpu()) < 1e-5


@pytest.mark.parametrize("nx,ny,B", [(16, 4, 5), (32, 32, 37), (64, 64, 130), (128, 16, 19), (128, 128, 64), (64, 2, 1)])
def test_one_kernel_route_for_many_weighting_functions(nx, ny, B, dev):
    """m > 32 on the reference's pixel meshes: vo_gridgemm.cuh (the fine residual produced inside the contraction kernel, zero
    tiles of V skipped) against the two-kernel route (rho through HBM + vo_gemm.cuh, GPDE_VO_GRIDGEMM=0) and the version-1
    kernels: both column-tile widths, several column tiles, sparse columns (tiles really get skipped), ragged batches,
    shared field / Dirichlet rows, no Dirichlet data, conductivity input, FP32 I/O, bitwise repeatability."""
    plan, fom, a, y, g, rng = _grid_case(nx, ny, "NDP", B, nx * 1000 + ny, dev, load=False)
    two, v1 = plan.variant(GPDE_VO_GRIDGEMM="0"), plan.variant(GPDE_VO_PATH="v1")
    T = lambda t: torch.tensor(t, device=dev)
    for m in (33, 70, 130, 256, 300):
        V = rng.normal(size=(fom.dim_out, m))
        V[:, : m // 3] *= rng.uniform(size=(fom.dim_out, m // 3)) < 0.02
        V = T(V)
        for kw in (dict(a=T(a), y=T(y), g=T(g)), dict(a=T(a[0]), y=T(y), g=T(g[0])),
                   dict(a=T(np.exp(a)), y=T(y), g=None, a_is_log=False)):
            r1 = plan.residual(V=V, **kw)
            assert rel_err(r1.cpu(), two.residual(V=V, **kw).cpu()) < 1e-12, (m, sorted(kw))
            assert torch.equal(r1, plan.residual(V=V, **kw))
        assert rel_err(plan.residual(T(a), T(y), T(g), V).cpu(), v1.residual(T(a), T(y), T(g), V).cpu()) < 1e-12, m
        f = lambda t: T(t).float()
        r32 = plan.residual(f(a), f(y), f(g), V.float())
        assert r32.dtype == torch.float32
        assert rel_err(r32.double().cpu(), two.residual(f(a), f(y), f(g), V.float()).double().cpu()) < 1e-5, m


@pytest.mark.parametrize("nx,ny,B", [(32, 32, 64), (32, 32, 5), (64, 64, 37), (16, 8, 130), (128, 16, 19), (64, 4, 3), (16, 2, 9)])
def test_small_batches_cut_the_node_rows_over_a_cluster(nx, ny, B, dev):
    """Few sample blocks: the lean grid kernel runs as thread-block clusters whose CTAs each march a range of the node
    rows (replaying the stage below their range) and meet through distributed shared memory (vo_grid2.cuh, SPLIT).
    Against one CTA per block (GPDE_GRID2_SPLIT=0) to summation-order rounding: automatic and forced cluster sizes, every
    n-tile split of m, FP64 and FP32 I/O (all phases of y), log and conductivity input, shared Dirichlet rows, packed
    weights; the cut does not depend on the position in the batch (bitwise sample-permutation equivariance)."""
    plan, fom, a, y, g, rng = _grid_case(nx, ny, "NDP", B, nx * 13 + ny + B, dev, load=False)
    whole = plan.variant(GPDE_GRID2_SPLIT="0")
    T = lambda t: torch.tensor(t, device=dev)
    d = fom.dim_out
    big = torch.zeros(B * d + 3, dtype=torch.float32, device=dev)
    y32_off = big[3:].view(B, d)
    y32_off.copy_(T(y).float())
    variants = [plan] + [plan.variant(GPDE_GRID2_SPLIT=str(c)) for c in (2, 3, 8)]     # the library caps the size at stages / 2
    for m in (1, 8, 9, 17, 25, 32):
        V = T(rng.normal(size=(d, m)))
        r0 = whole.residual(T(a), T(y), T(g), V)
        r0_lin = whole.residual(torch.exp(T(a)), T(y), T(g[0]), V, a_is_log=False)
        r0_32 = whole.residual(T(a).float(), y32_off, T(g).float(), V.float())
        for p in variants:
            assert rel_err(p.residual(T(a), T(y), T(g), V).cpu(), r0.cpu()) < 1e-12, m
            assert rel_err(p.residual(torch.exp(T(a)), T(y), T(g[0]), V, a_is_log=False).cpu(), r0_lin.cpu()) < 1e-12, m
            assert rel_err(p.residual(T(a).float(), y32_off, T(g).float(), V.float()).double().cpu(), r0_32.double().cpu()) < 2e-6, m
    V = T(rng.normal(size=(d, 25)))
    r = plan.residual(T(a), T(y), T(g), V)
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(0)).to(dev)
    assert torch.equal(plan.residual(T(a)[perm], T(y)[perm], T(g)[perm], V), r[perm])
    pw = plan.pack_weights(V, B)
    assert torch.equal(plan.residual(T(a), T(y), T(g), pw), r)


@pytest.mark.parametrize("nx,ny,B", [(64, 64, 229), (32, 32, 300), (16, 8, 700), (128, 16, 150), (64, 4, 163)])
def test_partly_filled_sample_groups_give_the_same_bits(nx, ny, B, dev):
    """The lean grid kernel fills the 8-sample groups of a CTA with fewer samples when that spreads the last wave of CTAs
    over all SMs (grid2_samples_per_cta in vo.cu: 4096 samples = 147 CTAs of 28 instead of 128 of 32).  A sample's
    arithmetic does not depend on its slot: every samples-per-CTA setting (forced through GPDE_GRID2_SPC, and the automatic
    one, with and without reserved SMs) must reproduce the full-group result BITWISE -- contraction and rho variants,
    FP64 and FP32 I/O at every phase of y, log and conductivity input, ragged last CTA."""
    plan, fom, a, y, g, rng = _grid_case(nx, ny, "NDP", B, nx * 7 + ny + B, dev, load=False)
    S = 8 * (16 // (nx // 16))
    full = plan.variant(GPDE_GRID2_SPLIT="0", GPDE_GRID2_SPC=str(S))
    T = lambda t: torch.tensor(t, device=dev)
    d = fom.dim_out
    big = torch.zeros(B * d + 3, dtype=torch.float32, device=dev)
    variants = [plan.variant(GPDE_GRID2_SPLIT="0", GPDE_GRID2_SPC=str(c)) for c in sorted({S - 1, S - 3, (7 * S) // 8, (3 * S) // 4})]
    variants.append(plan.variant(GPDE_GRID2_SPLIT="0"))
    for m in (8, 25, 32):
        V = T(rng.normal(size=(d, m)))
        r0 = full.residual(T(a), T(y), T(g), V)
        r0_lin = full.residual(torch.exp(T(a)), T(y), T(g[0]), V, a_is_log=False)
        _, rho0 = full.residual(torch.exp(T(a)), T(y), T(g[0]), None, a_is_log=False)
        for p in variants:
            assert torch.equal(p.residual(T(a), T(y), T(g), V), r0), m
            assert torch.equal(p.residual(torch.exp(T(a)), T(y), T(g[0]), V, a_is_log=False), r0_lin), m
            assert torch.equal(p.residual(torch.exp(T(a)), T(y), T(g[0]), None, a_is_log=False)[1], rho0), m
            assert torch.equal(p.residual(torch.exp(T(a)), T(y), T(g[0]), V, a_is_log=False, sm_reserve=11), r0_lin), m
        for off in range(4):
            y32 = big[off:off + B * d].view(B, d)
            y32.copy_(T(y).float())
            r0_32 = full.residual(T(a).float(), y32, T(g).float(), V.float())
            _, rho0_32 = full.residual(T(a).float(), y32, T(g).float(), None)
            for p in variants:
                assert torch.equal(p.residual(T(a).float(), y32, T(g).float(), V.float()), r0_32), (m, off)
                assert torch.equal(p.residual(T(a).float(), y32, T(g).float(), None)[1], rho0_32), (m, off)
    # against the version-1 kernels as an independent route
    V = T(rng.normal(size=(d, 25)))
    assert rel_err(variants[-1].residual(T(a), T(y), T(g), V).cpu(), plan.variant(GPDE_VO_PATH="v1").residual(T(a), T(y), T(g), V).cpu()) < 1e-11


@pytest.mark.parametrize("nx,ny,B", [(64, 64, 229), (32, 32, 70), (16, 8, 300), (16, 2, 9), (64, 4, 33), (128, 16, 21), (64, 2, 1)])
def test_transposed_application_in_one_kernel(nx, ny, B, dev):
    """q = K_ff(a) (V s) = Gamma^T s (VirtualObservables.py:663) with the rows of w = s V^T produced inside the marching
    kernel (WT variant of vo_grid2_kernel; w [B,d] never exists) against the two-kernel route (expansion kernel + marching
    kernel, GPDE_VO_FUSED_T=0) and the version-1 kernels: every k-step count (m <= 16, <= 28, <= 32), log and conductivity
    input, FP64 and FP32 I/O, ragged batches, partly filled sample groups; adjointness against the forward residual."""
    plan, fom, a, y, g, rng = _grid_case(nx, ny, "NDP", B, nx * 5 + ny + B, dev, load=False)
    two, v1 = plan.variant(GPDE_VO_FUSED_T="0"), plan.variant(GPDE_VO_PATH="v1")
    part = plan.variant(GPDE_GRID2_SPC=str(8 * (16 // (nx // 16)) - 3))
    T = lambda t: torch.tensor(t, device=dev)
    d = fom.dim_out
    for m in (1, 8, 16, 17, 25, 28, 32):
        V, sv = T(rng.normal(size=(d, m))), T(rng.normal(size=(B, m)))
        q = plan.residual_T(T(a), V, sv)
        assert rel_err(q.cpu(), two.residual_T(T(a), V, sv).cpu()) < 1e-12, m
        assert rel_err(q.cpu(), v1.residual_T(T(a), V, sv).cpu()) < 1e-11, m
        assert torch.equal(part.residual_T(T(a), V, sv), q), m
        q_lin = plan.residual_T(torch.exp(T(a)), V, sv, a_is_log=False)
        assert rel_err(q_lin.cpu(), q.cpu()) < 1e-12, m
        q32 = plan.residual_T(torch.exp(T(a)).float(), V.float(), sv.float(), a_is_log=False)
        assert q32.dtype == torch.float32
        assert rel_err(q32.double().cpu(), two.residual_T(torch.exp(T(a)).float(), V.float(), sv.float(), a_is_log=False).double().cpu()) < 2e-6, m
        assert rel_err(plan.residual_T(T(a).float(), V.float(), sv.float()).double().cpu(), q.cpu()) < 1e-5, m
    # sparse weighting functions: the kernel skips the 8-node x 4-function blocks of V that are zero (masks from the packing
    # kernel) -- bands of nodes per function (like the coarse mesh's hat functions), scattered entries, an all-zero V
    for m in (25, 32):
        sv = T(rng.normal(size=(B, m)))
        band = np.zeros((d, m))
        for j in range(m):
            lo = (j * d) // m
            band[lo:lo + max(1, d // 6), j] = rng.normal(size=min(d, lo + max(1, d // 6)) - lo)
        scattered = rng.normal(size=(d, m)) * (rng.uniform(size=(d, m)) < 0.02)
        for Vs in (band, scattered, np.zeros((d, m))):
            q = plan.residual_T(T(a), T(Vs), sv)
            q2 = two.residual_T(T(a), T(Vs), sv)
            assert torch.equal(q, q2) or rel_err(q.cpu(), q2.cpu()) < 1e-12, m
            assert torch.equal(part.residual_T(T(a), T(Vs), sv), q), m
    # <s, Gamma y> = <Gamma^T s, y> with zero Dirichlet data and no load
    V, sv = T(rng.normal(size=(d, 25))), T(rng.normal(size=(B, 25)))
    lhs = (plan.residual(T(a), T(y), None, V, ignore_load=True) * sv).sum(dim=1)
    rhs = (plan.residual_T(T(a), V, sv) * T(y)).sum(dim=1)
    assert rel_err(lhs.cpu(), rhs.cpu()) < 1e-11

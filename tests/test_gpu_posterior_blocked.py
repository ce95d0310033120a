"""Blocked, matrix-free posterior update for up to 256 virtual observables per data point (csrc/vo_posterior_blocked.cuh
through gpde_vo_posterior_blocked_f64) and the panel route of gpde_vo_moments_f64 for m > 64, against the oracle's
restatement of the reference's per-data-point arithmetic (oracle/vo_ref), the one-launch kernel for m <= 64 and the dense
route (condition_gaussian).  Tolerances as in test_gpu_posterior.py: 1e-9 on the mean, 1e-8 on the variances."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def _plan_and_oracle(nx, ny, dev):
    from oracle import fem_p1, vo_ref
    from gpde_b200 import fem
    from gpde_b200.physics import LinearEllipticPhysics
    from gpde_b200.VirtualObservables import VoPlan
    mesh = fem.P1Mesh(nx, ny)
    fom = LinearEllipticPhysics("fom", "NDP", mesh)
    plan = VoPlan(fom, dev, mesh.pixel_of_cell(), nx * ny)
    c, cells = fem_p1.unit_square_mesh(nx, ny)
    bc, _, free = fem_p1.dirichlet_left_right(c, "ND")
    return plan, fom, vo_ref.CsrAssembler(c, cells, bc, free), fem_p1.pixel_of_cell(c, cells, nx, ny), bc


def _problem(plan, fom, bc, nx, ny, m, N, shared, seed, dev, zeros=True):
    rng = np.random.RandomState(seed)
    d = fom.dim_out
    img = rng.normal(0.3, 0.7, size=(N, nx * ny))
    gbc = rng.uniform(-0.5, 0.5, size=(N, bc.size))
    V = rng.normal(size=(d, m)) if shared else rng.normal(size=(N, d, m))
    g = rng.normal(size=(N, d))
    prec = rng.uniform(0.5, 50.0, size=(N, d))
    noise = rng.uniform(1e-4, 1e-1, size=m)
    if zeros and m < d:
        noise[::3] = 0.0                  # infinite-precision observables (precision_mask = -1): Lambda stays SPD for m < d
    T = lambda t: torch.tensor(t, device=dev)
    a = torch.exp(T(img))
    _, rho = plan.residual(a, T(g), T(gbc), None, a_is_log=False)
    return dict(img=img, gbc=gbc, V=V, g=g, prec=prec, noise=noise, a=a, rho=rho,
                Vt=T(V), gt=T(g), pt=T(prec), nt=T(noise))


CASES = [(nx, ny, m) for nx, ny in ((8, 6), (16, 16), (32, 32)) for m in (1, 33, 64, 65, 100, 128, 129, 256)]


def _precision_form_posterior(Gam, alp, noise, g, prec):
    """The same posterior from the d x d precision matrix A = diag(prec) + Gamma^T diag(1/noise) Gamma (all noise > 0):
    vars = diag(A^-1), mean = A^-1 (prec g + Gamma^T (alpha / noise)).  For m >= d, Lambda = Gamma C Gamma^T + diag(noise) is
    conditioned by the noise alone, and vars = c - c^2 q^T Lambda^-1 q cancels to a few 1e-4 of c: the oracle's float64
    arithmetic (that same formula) is then off by up to ~5e-8, while this form stays within ~1e-12 of a 40-digit
    evaluation (test_precision_form_reference_is_accurate)."""
    Gam, alp, noise, g, prec = (torch.as_tensor(t, dtype=torch.float64) for t in (Gam, alp, noise, g, prec))
    A = Gam.t() @ (Gam / noise[:, None]) + torch.diag(prec)
    Li = torch.linalg.solve_triangular(torch.linalg.cholesky(A), torch.eye(A.shape[0], dtype=torch.float64), upper=False)
    return Li.t() @ (Li @ (prec * g + Gam.t() @ (alp / noise))), (Li ** 2).sum(0)


def _reference(Gam, alp, noise, g, prec):
    """(mean, vars, tol_mean, tol_vars): the oracle at 1e-9 / 1e-8 where Lambda is well conditioned (m < d); for m >= d
    the precision form, with 1e-9 / 1e-8 or ten times the oracle's own error on the same instance, whichever is larger."""
    from oracle import vo_ref
    mean0, vars0 = vo_ref.virtual_observable_update(Gam, alp, noise, g, prec)
    if Gam.shape[0] < Gam.shape[1]:
        return mean0, vars0, 1e-9, 1e-8
    mean1, vars1 = _precision_form_posterior(Gam, alp, noise, g, prec)
    return mean1, vars1, max(1e-9, 10 * rel_err(mean0, mean1)), max(1e-8, 10 * rel_err(vars0, vars1))


def test_precision_form_reference_is_accurate():
    """The float64 precision form against 40-digit arithmetic (mpmath) on a rank-deficient instance of the oracle test."""
    import mpmath
    from oracle import fem_p1, vo_ref
    c, cells = fem_p1.unit_square_mesh(8, 6)
    bc, _, free = fem_p1.dirichlet_left_right(c, "ND")
    asm, pix = vo_ref.CsrAssembler(c, cells, bc, free), fem_p1.pixel_of_cell(c, cells, 8, 6)
    rng = np.random.RandomState(3)
    d, m = free.size, 100
    K, f = asm.assemble(np.exp(rng.normal(0.3, 0.7, size=48))[pix], rng.uniform(-0.5, 0.5, size=bc.size))
    Gam, alp = (np.asarray(t) for t in vo_ref.construct_querry_weak_galerkin(K, f, rng.normal(size=(d, m))))
    g, prec, noise = rng.normal(size=d), rng.uniform(0.5, 50.0, size=d), rng.uniform(1e-4, 1e-1, size=m)
    mean1, vars1 = _precision_form_posterior(Gam, alp, noise, g, prec)
    with mpmath.workdps(40):
        G = mpmath.matrix(Gam.tolist())
        GtN = G.T * mpmath.diag([1 / mpmath.mpf(x) for x in noise])
        A = GtN * G
        for i in range(d):
            A[i, i] += mpmath.mpf(prec[i])
        S = mpmath.inverse(A)
        mhp = S * (mpmath.matrix([mpmath.mpf(prec[i]) * g[i] for i in range(d)]) + GtN * mpmath.matrix(alp.tolist()))
        mean_hp, vars_hp = np.array([float(x) for x in mhp]), np.array([float(S[i, i]) for i in range(d)])
    assert rel_err(mean1, mean_hp) < 1e-11 and rel_err(vars1, vars_hp) < 1e-11


@pytest.mark.parametrize("nx,ny,m", CASES)
def test_posterior_blocked_matches_oracle(nx, ny, m, dev):
    from oracle import vo_ref
    plan, fom, asm, pix, bc = _plan_and_oracle(nx, ny, dev)
    k = CASES.index((nx, ny, m))
    N, shared = (1, 3, 7)[k % 3], bool(k % 2)
    p = _problem(plan, fom, bc, nx, ny, m, N, shared, 1000 + k, dev)
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    mean, vars_ = plan.posterior_blocked(p["a"], p["Vt"], p["rho"], p["nt"], p["gt"], p["pt"], info=info)
    assert int(info.item()) == 0
    r_k, s2_k = plan.moments(p["a"], p["Vt"], p["rho"], torch.tensor(1.0 / p["prec"], device=dev))
    for n in range(N):
        K, f = asm.assemble(np.exp(p["img"][n][pix]), p["gbc"][n])
        Vn = p["V"] if shared else p["V"][n]
        Gam, alp = vo_ref.construct_querry_weak_galerkin(K, f, Vn)
        mean0, vars0, tol_mean, tol_vars = _reference(Gam, alp, p["noise"], p["g"][n], p["prec"][n])
        assert rel_err(mean[n].cpu(), mean0) < tol_mean, (n, rel_err(mean[n].cpu(), mean0), tol_mean)
        assert rel_err(vars_[n].cpu(), vars0) < tol_vars, (n, rel_err(vars_[n].cpu(), vars0), tol_vars)
        assert rel_err(r_k[n].cpu(), Gam @ p["g"][n] - alp) < 1e-10, n
        assert rel_err(s2_k[n].cpu(), (Gam ** 2) @ (1.0 / p["prec"][n])) < 1e-10, n
    if m <= 64:        # the one-launch kernel on the same inputs
        mean1, vars1 = plan.posterior(p["a"], p["Vt"], p["rho"], p["nt"], p["gt"], p["pt"])
        tol = 1e-11
        if m >= fom.dim_out:
            # Gamma C Gamma^T has rank d < m: Lambda is conditioned by the noise variances alone (cond ~ 1e6 here), and
            # the two kernels' different summation orders differ by up to ~eps cond
            for n in range(N):
                K, f = asm.assemble(np.exp(p["img"][n][pix]), p["gbc"][n])
                Gam = torch.as_tensor(vo_ref.construct_querry_weak_galerkin(K, f, p["V"] if shared else p["V"][n])[0])
                Lam = (Gam / torch.tensor(p["prec"][n])) @ Gam.t() + torch.diag(torch.tensor(p["noise"]))
                tol = max(tol, 10 * np.finfo(np.float64).eps * float(torch.linalg.cond(Lam)))
        assert rel_err(mean.cpu(), mean1.cpu()) < tol
        assert rel_err(vars_.cpu(), vars1.cpu()) < tol


def test_posterior_blocked_config3_shape_against_dense_conditioning(dev):
    """128 x 128 mesh, m = 256 = W (81 columns) + 175 RBF columns (l = 0.1), N = 4: against condition_gaussian on the
    materialised Gamma_n, with a tolerance from the condition number of Lambda_n."""
    from gpde_b200.VirtualObservables import VoPlan, condition_gaussian
    from gpde_b200.workloads import Workload
    w = Workload("cfg3", B=4, seed=3)
    fom = w.physics["fom"]
    plan = VoPlan.cached(fom, dev, pixel_input=True)
    N, d, m = 4, w.d, w.m
    assert m == 256
    rng = np.random.RandomState(5)
    T = lambda t: torch.tensor(t, device=dev)
    a = torch.exp(T(w.log_image))
    V, gbc = T(w.V), T(w.g_fom)
    g, prec = T(rng.normal(size=(N, d))), T(rng.uniform(0.5, 50.0, size=(N, d)))
    noise = T(rng.uniform(1e-4, 1e-1, size=m))
    _, rho = plan.residual(a, g, gbc, None, a_is_log=False)
    mean, vars_ = plan.posterior_blocked(a, V, rho, noise, g, prec)
    eye = torch.eye(m, dtype=torch.float64, device=dev)
    for n in range(N):
        Gam = plan.residual_T(a[n:n + 1].expand(m, -1).contiguous(), V, eye, a_is_log=False)       # [m,d]: rows Gamma^T e_j
        r = plan.residual(a[n:n + 1], g[n:n + 1], gbc[n:n + 1], V, a_is_log=False)[0]
        alp = Gam @ g[n] - r
        mean0, vars0 = condition_gaussian(Gam[None], alp[None], noise, g[n:n + 1], prec[n:n + 1])
        Lam = (Gam / prec[n]) @ Gam.t() + torch.diag(noise)
        cond = float(torch.linalg.cond(Lam).item())
        tol = max(1e-12, 1e3 * np.finfo(np.float64).eps * cond)
        assert rel_err(mean[n].cpu(), mean0[0].cpu()) < tol, (n, cond)
        assert rel_err(vars_[n].cpu(), vars0[0].cpu()) < 10 * tol, (n, cond)


def test_posterior_blocked_row_split_matches_unsplit_call(dev):
    """N = 1 at m = 256 splits the Gram pass over row segments (its workspace holds the partial blocks); the same data
    point inside a batch of 64 runs unsplit."""
    nx = ny = 32
    plan, fom, asm, pix, bc = _plan_and_oracle(nx, ny, dev)
    m, N = 256, 64
    p = _problem(plan, fom, bc, nx, ny, m, N, False, 7, dev)
    assert plan.posterior_blocked_workspace_bytes(1, m) > plan.posterior_blocked_workspace_bytes(N, m) // N
    mean, vars_ = plan.posterior_blocked(p["a"], p["Vt"], p["rho"], p["nt"], p["gt"], p["pt"])
    for n in (0, 17):
        sl = slice(n, n + 1)
        m1, v1 = plan.posterior_blocked(p["a"][sl], p["Vt"][sl], p["rho"][sl], p["nt"], p["gt"][sl], p["pt"][sl])
        assert rel_err(m1[0].cpu(), mean[n].cpu()) < 1e-13
        assert rel_err(v1[0].cpu(), vars_[n].cpu()) < 1e-13


@pytest.mark.parametrize("m", [100, 256])
def test_posterior_blocked_is_deterministic(m, dev):
    nx = ny = 16
    plan, fom, asm, pix, bc = _plan_and_oracle(nx, ny, dev)
    N = 6
    p = _problem(plan, fom, bc, nx, ny, m, N, True, 11, dev)
    args = (p["a"], p["Vt"], p["rho"], p["nt"], p["gt"], p["pt"])
    mean, vars_ = plan.posterior_blocked(*args)
    for _ in range(3):
        m2, v2 = plan.posterior_blocked(*args)
        assert torch.equal(m2, mean) and torch.equal(v2, vars_)
    perm = torch.tensor([3, 0, 5, 1, 4, 2], device=dev)
    mp_, vp_ = plan.posterior_blocked(p["a"][perm], p["Vt"], p["rho"][perm], p["nt"], p["gt"][perm], p["pt"][perm])
    assert torch.equal(mp_, mean[perm]) and torch.equal(vp_, vars_[perm])


def test_posterior_blocked_errors(dev):
    from gpde_b200 import _lib
    nx = ny = 16
    plan, fom, asm, pix, bc = _plan_and_oracle(nx, ny, dev)
    m, N = 100, 3
    p = _problem(plan, fom, bc, nx, ny, m, N, True, 13, dev)
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    plan.posterior_blocked(p["a"], p["Vt"], p["rho"], torch.full((m,), -1e9, dtype=torch.float64, device=dev),
                           p["gt"], p["pt"], info=info)
    assert int(info.item()) == 2
    lib, P = plan._lib, lambda t: _lib.ptr(t, dev)
    mean, vars_ = torch.zeros_like(p["gt"]), torch.zeros_like(p["gt"])
    need = plan.posterior_blocked_workspace_bytes(N, m)
    ws = torch.zeros(need + 64, dtype=torch.uint8, device=dev)
    st = _lib.stream_of(dev)

    def call(V, mm, wsp, nbytes, n=N):
        return lib.gpde_vo_posterior_blocked_f64(plan.handle, P(p["a"]), plan.n_inputs, P(V), 0, mm, P(p["rho"]),
                                                 P(p["nt"]), P(p["gt"]), P(p["pt"]), P(mean), P(vars_), None, wsp,
                                                 nbytes, n, st)
    V257 = torch.zeros(fom.dim_out, 257, dtype=torch.float64, device=dev)
    assert call(V257, 257, P(ws), ws.numel()) == -3                                  # GPDE_ERR_SIZE
    assert call(p["Vt"], m, None, need) == -1                                         # GPDE_ERR_ARG: null
    assert call(p["Vt"], m, ctypes.c_void_p(ws.data_ptr() + 8), need) == -1           # misaligned
    assert call(p["Vt"], m, P(ws), need - 8) == -1                                    # too small
    assert call(p["Vt"], m, P(ws), 0, n=0) == 0                                       # N = 0: nothing to do
    torch.cuda.synchronize()
    assert not mean.any() and not vars_.any()
    assert call(p["Vt"], m, P(ws), need) == 0
    torch.cuda.synchronize()
    assert torch.isfinite(mean).all() and torch.isfinite(vars_).all()
    with pytest.raises(Exception):
        plan.posterior_blocked(p["a"], V257, p["rho"], torch.ones(257, dtype=torch.float64, device=dev), p["gt"], p["pt"])


def _ensemble(dev, N, extra_rbf, seed=4, learnable=True):
    """32 x 32 fine mesh, V = W (25 columns) + ``extra_rbf`` RBF columns per data point."""
    from gpde_b200 import VirtualObservables as VO
    from gpde_b200.physics import setup_physics, BoundaryConditionEnsemble
    from gpde_b200 import fem
    rng = np.random.RandomState(seed)
    ph = setup_physics(4, 4, 3, "NDP")
    fom = ph['fom']
    img = fem.sample_log_field(32, 32, 0.4, 0.8, 0.15, N, rng)
    X_DG = img.reshape(N, -1)[:, fom.mesh.pixel_of_cell()]
    bce = BoundaryConditionEnsemble(ph, N, "NDP", rng=rng)
    qpe = VO.QuerryPointEnsemble.FromArrays(X_DG, bce, fom, device=dev)
    np.random.seed(seed)
    qe = VO.QuerryEnsemble.FromQuerryPointEnsemble(qpe, ph, CGR=True, flux=False, N_gaussian=0, N_rbf=extra_rbf, l_rbf=0.2,
                                                   dtype=torch.double, device=dev)
    if learnable:
        for q in qe:
            q._sampler.__class__ = type("Learnable", (q._sampler.__class__,), {"precision_mask": property(lambda s: np.ones(s.m))})
    ens = VO.VirtualObservablesEnsemble(qpe, qe, torch.double, dev)
    return ph, ens, qe, X_DG, bce, rng


@pytest.mark.parametrize("extra_rbf", [45, 175])
def test_ensemble_blocked_route_matches_oracle_loop(extra_rbf, dev):
    from oracle import fem_p1, vo_ref
    ph, ens, qe, X_DG, bce, rng = _ensemble(dev, 5, extra_rbf)
    N, d, m = ens.N, ens.dim_out, ens.m
    assert m == 25 + extra_rbf
    T = lambda t: torch.tensor(t, device=dev)
    G1, P1 = rng.normal(size=(N, d)), rng.uniform(1.0, 30.0, size=(N, d))
    G2, P2 = rng.normal(size=(N, d)), rng.uniform(1.0, 30.0, size=(N, d))
    ens.update(T(G1), T(P1), 0)
    ens.check()
    assert ens.last_update_route == "blocked"
    m1, v1 = ens.mean.clone(), ens.vars.clone()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ens.update(T(G2), T(P2), 1)                                 # includes the precision hyper-update on (m1, v1)
        torch.cuda.synchronize()
    assert ens.last_update_route == "blocked"
    assert all("Gamma" not in q._store for q in qe)
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    for k in ("vo_post_gram_kernel", "vo_post_factor_kernel", "vo_post_apply_kernel", "vo_moments_panel_kernel"):
        assert any(k in s for s in names), k
    vendor = ("cublas", "cusolver", "potrf", "trsm", "syrk", "gemm", "xmma", "cutlass", "magma")
    assert not [s for s in names if "gpde" not in s and any(v in s.lower() for v in vendor)]
    # oracle: the reference's loop over data points on dense Gamma
    P = fem_p1.build_problem(4, 4, 3)
    Gams, alps = [], []
    for n in range(N):
        K, f = fem_p1.assemble_system_free(P['coords_fom'], P['cells_fom'], np.exp(X_DG[n]), P['bc_dofs_fom'],
                                           bce[n].constrained_dofs_values('fom'), P['free_dofs_fom'])
        Gam, alp = vo_ref.construct_querry_weak_galerkin(K, f, qe[n].V.cpu().numpy())
        Gams.append(Gam); alps.append(alp)
    prec_alpha = 0.5 * N + 1e-6
    mask = torch.zeros(m, dtype=torch.bool)
    var0 = vo_ref.mean_vo_variances(torch.ones(m, dtype=torch.double), prec_alpha, mask)
    post1 = [vo_ref.virtual_observable_update(Gams[n], alps[n], var0, G1[n], P1[n]) for n in range(N)]
    assert rel_err(m1.cpu(), torch.stack([p[0] for p in post1])) < 1e-9
    assert rel_err(v1.cpu(), torch.stack([p[1] for p in post1])) < 1e-8
    beta = vo_ref.update_vo_precision_beta(Gams, alps, [p[0] for p in post1], [p[1] for p in post1])
    assert rel_err(ens._prec_beta.cpu(), beta) < 1e-8
    var1 = vo_ref.mean_vo_variances(beta, prec_alpha, mask)
    post2 = [vo_ref.virtual_observable_update(Gams[n], alps[n], var1, G2[n], P2[n]) for n in range(N)]
    assert rel_err(ens.mean.cpu(), torch.stack([p[0] for p in post2])) < 1e-8
    assert rel_err(ens.vars.cpu(), torch.stack([p[1] for p in post2])) < 1e-7


def test_ensemble_routes_and_chunking(dev):
    from gpde_b200 import VirtualObservables as VO
    ph, ens, qe, X_DG, bce, rng = _ensemble(dev, 5, 45, seed=6)
    N, d = ens.N, ens.dim_out
    T = lambda t: torch.tensor(t, device=dev)
    G, P = T(rng.normal(size=(N, d))), T(rng.uniform(1.0, 30.0, size=(N, d)))
    ens.update(G, P, 0)
    assert ens.last_update_route == "blocked"
    mean, vars_ = ens.mean.clone(), ens.vars.clone()
    # the workspace budget cuts the data points into chunks; the chunks use their own row split (within 1e-13)
    plan = ens._inputs()[0]
    ens.max_stack_bytes = 2 * plan.posterior_blocked_workspace_bytes(1, ens.m)
    ens._precision_initialized = False          # skip the hyper-update: condition on the same noise variances again
    ens.update(G, P, 0)
    assert ens.last_update_route == "blocked"
    assert rel_err(ens.mean.cpu(), mean.cpu()) < 1e-13 and rel_err(ens.vars.cpu(), vars_.cpu()) < 1e-13
    del ens.max_stack_bytes
    # max_blocked_m on the instance forces the dense route
    ens.max_blocked_m = 64
    ens._precision_initialized = False
    ens.update(G, P, 0)
    assert ens.last_update_route == "dense"
    assert rel_err(ens.mean.cpu(), mean.cpu()) < 1e-9 and rel_err(ens.vars.cpu(), vars_.cpu()) < 1e-8
    # m <= 64: the one-launch kernel
    ph2, ens2, *_ = _ensemble(dev, 3, 4, seed=8)
    ens2.update(T(rng.normal(size=(3, d))), T(rng.uniform(1.0, 30.0, size=(3, d))), 0)
    assert ens2.last_update_route == "kernel"
    # a Lambda that is not positive definite: the info word is set and check() raises
    ph3, ens3, *_ = _ensemble(dev, 3, 45, seed=9, learnable=False)
    ens3._mean_vo_variances = torch.full((ens3.m,), -1e9, dtype=torch.float64, device=dev)
    ens3.update(T(rng.normal(size=(3, d))), T(rng.uniform(1.0, 30.0, size=(3, d))), 0)
    assert ens3.last_update_route == "blocked"
    with pytest.raises(RuntimeError):
        ens3.check()
    ens3.check()                                                    # cleared


def test_flux_ensemble_stays_dense(dev):
    from gpde_b200 import VirtualObservables as VO
    from gpde_b200.physics import BoundaryConditionEnsemble, setup_physics
    ph = setup_physics(2, 2, 2, "NDP")
    fom = ph['fom']
    rng = np.random.RandomState(3)
    N = 3
    X = rng.normal(0.4, 0.8, size=(N, fom.dim_in))
    bce = BoundaryConditionEnsemble(ph, N, "NDP", rng=rng)
    qpe = VO.QuerryPointEnsemble.FromArrays(X, bce, fom, device=dev)
    qe = VO.QuerryEnsemble.FromQuerryPointEnsemble(qpe, ph, True, True, 0, 0, dtype=torch.float64, device=dev)
    ens = VO.VirtualObservablesEnsemble(qpe, qe, dtype=torch.float64, device=dev)
    G = torch.tensor(rng.normal(size=(N, fom.dim_out)), device=dev)
    P = torch.tensor(rng.uniform(0.5, 2.0, size=(N, fom.dim_out)), device=dev)
    ens.update(G, P, 0)
    assert ens.last_update_route == "dense"

"""Batched subspace-Newton step of the energy-type virtual observables (csrc/vo_energy.cuh through the C ABI) and the batched
route of EnergyVirtualObservablesEnsemble.update:
    kernel        rho launch + gpde_vo_energy_step_f64, repeated   -> oracle/vo_ref.energy_vo_update per data point (1e-10)
    ensemble      batched route against the member loop (EnergyVirtualObservable.update per data point) on the same draws
"""
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


def _kernel_case(nx, ny, kind, N, seed, dev):
    from oracle import fem_p1, vo_ref
    from gpde_b200 import fem
    from gpde_b200.physics import LinearEllipticPhysics
    from gpde_b200.VirtualObservables import VoPlan
    rng = np.random.RandomState(seed)
    mesh = fem.P1Mesh(nx, ny)
    fom = LinearEllipticPhysics("fom", kind, mesh)
    plan = VoPlan(fom, dev)
    c, cells = fem_p1.unit_square_mesh(nx, ny)
    bc, _, free = fem_p1.dirichlet_left_right(c, "ND")
    asm = vo_ref.CsrAssembler(c, cells, bc, free)
    if kind == "ND":
        gbc = np.tile(mesh.dirichlet_values("ND")[None], (N, 1))
    else:
        gbc = np.atleast_2d(mesh.dirichlet_values("NDP", rng.uniform(-0.5, 0.5, size=(N, 4))))
    return plan, fom, asm, gbc, rng


@pytest.mark.parametrize("nx,ny,kind,m,N,shared_V,shared_a", [
    (4, 4, "ND", 1, 7, True, False),
    (8, 6, "NDP", 40, 5, False, False),
    (16, 16, "NDP", 6, 5, True, True),
    (16, 16, "ND", 32, 7, False, False),
    (32, 32, "NDP", 64, 1, True, False),
    (16, 16, "NDP", 64, 5, False, True),
])
def test_energy_step_kernel_matches_oracle(nx, ny, kind, m, N, shared_V, shared_a, dev):
    from oracle import vo_ref
    plan, fom, asm, gbc, rng = _kernel_case(nx, ny, kind, N, nx * 100 + m, dev)
    d, n_steps = fom.dim_out, 3
    x = rng.normal(0.2, 0.6, size=(1 if shared_a else N, fom.dim_in))
    g = rng.normal(size=(N, d))
    prec = rng.uniform(0.5, 50.0, size=(N, d))
    T_n = rng.uniform(0.05, 2.0, size=N)                                  # a different temperature per data point
    mean0 = rng.normal(size=(N, d))                                       # warm start
    Vs = [rng.normal(size=(d, m)) if shared_V else rng.normal(size=(N, d, m)) for _ in range(n_steps)]
    Tt = lambda t: torch.tensor(t, device=dev)
    a = torch.exp(Tt(x[0] if shared_a else x))
    gbc_t = Tt(gbc)
    mean = Tt(mean0).clone()
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    for V in Vs:
        _, rho = plan.residual(a, mean, gbc_t, None, a_is_log=False)
        out = plan.energy_step(a, Tt(V), rho, Tt(g), Tt(prec), Tt(1.0 / T_n), mean, info=info)
        assert out is mean
    assert int(info.item()) == 0
    for n in range(N):
        K, f = asm.assemble(np.exp(x[0 if shared_a else n]), gbc[n])
        want, _ = vo_ref.energy_vo_update(K, f, g[n], prec[n], mean0[n], [V if shared_V else V[n] for V in Vs], T_n[n])
        assert rel_err(mean[n].cpu(), want) < 1e-10, n


def test_energy_step_limits_and_info_word(dev):
    plan, fom, asm, gbc, rng = _kernel_case(16, 16, "NDP", 3, 5, dev)
    N, d = 3, fom.dim_out
    Tt = lambda t: torch.tensor(t, device=dev)
    a = torch.exp(Tt(rng.normal(size=(N, fom.dim_in))))
    g, mean = Tt(rng.normal(size=(N, d))), Tt(rng.normal(size=(N, d)))
    prec, inv_T = Tt(rng.uniform(1.0, 10.0, size=(N, d))), Tt(np.ones(N))
    _, rho = plan.residual(a, mean, Tt(gbc), None, a_is_log=False)
    with pytest.raises(RuntimeError):                                      # m = 65: GPDE_ERR_SIZE
        plan.energy_step(a, Tt(rng.normal(size=(d, 65))), rho, g, prec, inv_T, mean)
    # a strongly negative precision on data point 1 makes its M indefinite: info word, mean kept, no trap
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    prec_bad = prec.clone()
    prec_bad[1] = -1e6
    before = mean.clone()
    plan.energy_step(a, Tt(rng.normal(size=(d, 6))), rho, g, prec_bad, inv_T, mean, info=info)
    assert int(info.item()) == 2
    assert torch.equal(mean[1], before[1]) and not torch.equal(mean[0], before[0])


# ------------------------------------------------------------------------------------------------ ensemble
def _ensemble(dev, N=5, n_it=3, sampler=None, seed=4):
    from gpde_b200 import VirtualObservables as VO
    from gpde_b200.physics import setup_physics, BoundaryConditionEnsemble
    rng = np.random.RandomState(seed)
    ph = setup_physics(2, 2, 3, "NDP")                                     # 16 x 16 fine mesh, d = 255
    fom = ph['fom']
    bce = BoundaryConditionEnsemble(ph, N, "NDP", rng=rng)
    qpe = VO.QuerryPointEnsemble.FromArrays(rng.normal(0.0, 0.5, size=(N, fom.dim_in)), bce, fom, device=dev)
    ens = VO.EnergyVirtualObservablesEnsemble(qpe, n_it, sampler(qpe) if sampler else None, torch.double, dev)
    ens.set_linear_temperature_schedule(T_init=1.0, T_final=1e-2, num_steps=4)
    return ens, fom


def _recording_sampler(m, seed):
    from gpde_b200 import VirtualObservables as VO

    class Recording(VO.BaseSampler):
        """Draw k is a seeded matrix whose first entry is k: the record shows which draw went where."""

        def __init__(self, qp):
            super().__init__(qp)
            self.rng, self.calls = np.random.RandomState(seed), 0

        def _sample(self):
            V = self.rng.normal(size=(self.qp.dim_out, m))
            V[0, 0] = self.calls
            self.calls += 1
            return V
    return Recording


def _inputs(fom, N, seed):
    rng = np.random.RandomState(seed)
    return [(rng.normal(size=(N, fom.dim_out)), rng.uniform(1.0, 30.0, size=(N, fom.dim_out))) for _ in range(3)]


def _run(ens, inputs, dev):
    out = []
    for it, (G, P) in enumerate(inputs):
        ens.update(torch.tensor(G, device=dev), torch.tensor(P, device=dev), it)
        out.append((ens.mean.clone(), ens.vars.clone(), [vo.temperature for vo in ens]))
    return out


def _assert_same(out_a, out_b):
    for (ma, va, ta), (mb, vb, tb) in zip(out_a, out_b):
        assert rel_err(ma.cpu(), mb.cpu()) < 1e-10
        assert torch.equal(va, vb)
        assert ta == tb


def test_batched_route_matches_member_loop_with_a_shared_recording_sampler(dev):
    Rec = _recording_sampler(6, 11)
    samplers = []

    def make(qpe):
        samplers.append(Rec(qpe[0]))
        return samplers[-1]

    ens_b, fom = _ensemble(dev, sampler=make)
    ens_m, _ = _ensemble(dev, sampler=make)
    ens_m.batched_update = False
    # the member loop draws data point-major, iteration-minor: record which draw each (data point, iteration) receives
    order = []
    for n, vo in enumerate(ens_m):
        def wrapped(n=n, s=vo._sampler):
            V = Rec._sample(s)
            order.append((n, float(V[0, 0])))
            return V
        vo._sampler = type("Tap", (), {"sample_V": staticmethod(wrapped), "m": 6})()
    inputs = _inputs(fom, ens_b.N, 2)
    out_b, out_m = _run(ens_b, inputs, dev), _run(ens_m, inputs, dev)
    assert ens_b.last_update_route == "batched" and ens_m.last_update_route == "members"
    assert samplers[0].calls == samplers[1].calls == 3 * ens_b.N * 3
    n_it, N = 3, ens_b.N
    assert order == [(n, float(u * N * n_it + n * n_it + k)) for u in range(3) for n in range(N) for k in range(n_it)]
    _assert_same(out_b, out_m)


@pytest.mark.parametrize("shared", [True, False])
def test_batched_route_matches_member_loop_with_seeded_rbf_samplers(shared, dev):
    from gpde_b200 import VirtualObservables as VO
    make = lambda qpe: VO.RadialBasisFunctionSampler(qpe[0], 0.3, 8)
    outs = []
    for batched in (True, False):
        ens, fom = _ensemble(dev, sampler=make)
        if not shared:           # one sampler per data point: drawn member by member, then concatenated
            for vo in ens:
                vo._sampler = VO.RadialBasisFunctionSampler(vo.querry_point, 0.3, 8)
        ens.batched_update = batched
        np.random.seed(21)
        outs.append(_run(ens, _inputs(fom, ens.N, 3), dev))
        assert ens.last_update_route == ("batched" if batched else "members")
    _assert_same(*outs)


def test_chunking_and_members(dev):
    from gpde_b200 import VirtualObservables as VO
    make = lambda qpe: VO.RadialBasisFunctionSampler(qpe[0], 0.3, 8)
    ens1, fom = _ensemble(dev, sampler=make)
    ens2, _ = _ensemble(dev, sampler=make)
    ens2.max_stack_bytes = 1                                               # one data point per chunk
    inputs = _inputs(fom, ens1.N, 5)
    np.random.seed(8)
    out1 = _run(ens1, inputs, dev)
    np.random.seed(8)
    out2 = _run(ens2, inputs, dev)
    for (m1, v1, _), (m2, v2, _) in zip(out1, out2):
        assert rel_err(m2.cpu(), m1.cpu()) < 1e-12 and torch.equal(v1, v2)
    # members read their rows of the batched result
    for n, vo in enumerate(ens1):
        assert torch.equal(vo.mean, ens1.mean[n]) and torch.equal(vo.vars, ens1.vars[n])
    # a member updated on its own afterwards: the same as that member in a member-loop ensemble in the same state
    ens3, _ = _ensemble(dev, sampler=make)
    ens3.batched_update = False
    np.random.seed(8)
    _run(ens3, inputs, dev)
    others = ens1.mean.clone()
    G, P = (torch.tensor(t[2], device=dev) for t in inputs[0])
    np.random.seed(9)
    ens1[2].update(G, P, 2, ForceUpdate=True)
    np.random.seed(9)
    ens3[2].update(G, P, 2, ForceUpdate=True)
    assert rel_err(ens1[2].mean.cpu(), ens3[2].mean.cpu()) < 1e-10
    ens1.flush_cache()
    assert torch.equal(ens1.mean[2], ens1[2].mean)
    assert torch.equal(ens1.mean[[0, 1, 3, 4]], others[[0, 1, 3, 4]])


def test_indefinite_newton_matrix_raises(dev):
    from gpde_b200 import VirtualObservables as VO
    ens, fom = _ensemble(dev, sampler=lambda qpe: VO.RadialBasisFunctionSampler(qpe[0], 0.3, 8))
    N, d = ens.N, fom.dim_out
    G = torch.zeros(N, d, dtype=torch.double, device=dev)
    P = torch.full((N, d), -1e6, dtype=torch.double, device=dev)
    with pytest.raises(RuntimeError):
        ens.update(G, P, 0)
    assert ens[0].mean is None                                             # nothing was committed
    ens.update(G, torch.ones(N, d, dtype=torch.double, device=dev), 1)     # the info word was cleared
    assert ens.last_update_route == "batched"


def test_member_loop_fallbacks(dev):
    from gpde_b200 import VirtualObservables as VO
    # m > 64 announced by the sampler: member loop, nothing drawn by the batched route
    ens, fom = _ensemble(dev, n_it=1, sampler=lambda qpe: VO.RadialBasisFunctionSampler(qpe[0], 0.3, 70))
    inputs = _inputs(fom, ens.N, 6)[:1]
    _run(ens, inputs, dev)
    assert ens.last_update_route == "members"
    # m > 64 found only in the draws (no ``m`` attribute): the member loop runs on the draws already made, in order
    Rec = _recording_sampler(70, 12)
    outs = []
    for batched in (True, False):
        ens, _ = _ensemble(dev, n_it=2, sampler=lambda qpe: Rec(qpe[0]))
        ens.batched_update = batched
        outs.append(_run(ens, inputs, dev))
        assert ens.last_update_route == "members" and ens[0]._sampler.calls == 2 * ens.N
        assert all(isinstance(vo._sampler, Rec) for vo in ens)             # the members' samplers are restored
    _assert_same(*outs)
    # members that differ in iterations per update
    ens, _ = _ensemble(dev, sampler=lambda qpe: VO.RadialBasisFunctionSampler(qpe[0], 0.3, 8))
    ens[1]._num_iterations_per_update = 2
    _run(ens, inputs, dev)
    assert ens.last_update_route == "members"

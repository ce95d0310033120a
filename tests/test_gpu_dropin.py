"""Drop-in proof for the callers of the hot path (VERDICT r1, item 1b): the ELBO of the reference's GenerativeModel
(bottleneck/generative.py:247-287, 352-392, 456-500) evaluated around the MIRRORED modules -- ROM, ReducedOrderModelOperator,
QuerryPointEnsemble / QuerryEnsemble / VirtualObservablesEnsemble of this package, running the sm_100a kernels -- reproduces
the value and all parameter gradients that the UNMODIFIED reference classes produced (tests/golden/elbo_4x4_16_ndp.npz).

The reference's sources are not part of this repository, so the caller's code is the restatement in oracle/elbo_ref.py;
tests/test_oracle_golden.py::test_elbo_restatement_matches_reference_generative_model pins that restatement to the values the
real GenerativeModel stored in the same fixture."""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_err
import elbo_fixture

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def _mirrors(G, dtype, dev):
    from gpde_b200 import VirtualObservables as VO
    from gpde_b200.components import ReducedOrderModelOperator
    from gpde_b200.physics import setup_physics, BoundaryConditionEnsemble
    ph = setup_physics(int(G['nx']), int(G['nx']), int(G['refines']), str(G['kind']))
    g = ReducedOrderModelOperator.FromPhysics(ph, dtype=dtype, device=dev)
    Nvo = G['in_vo_X_DG'].shape[0]
    bce = BoundaryConditionEnsemble(ph, Nvo, str(G['kind']), coefficients=G['in_vo_bc_coef'])
    assert np.allclose(bce.constrained_dofs_values('fom'), G['in_vo_g_fom'], atol=1e-15)
    qpe = VO.QuerryPointEnsemble.FromArrays(G['in_vo_X_DG'], bce, ph['fom'], device=dev)
    qe = VO.QuerryEnsemble.FromQuerryPointEnsemble(qpe, ph, CGR=True, flux=False, N_gaussian=0, N_rbf=0, dtype=torch.double,
                                                   device=dev)
    ens = VO.VirtualObservablesEnsemble(qpe, qe, dtype, dev)
    ens.update(torch.tensor(G['in_vo_G'], device=dev), torch.tensor(G['in_vo_PREC'], device=dev), 0)
    ens.check()
    return ph, g, ens


def test_reference_elbo_and_gradients_on_the_mirrored_modules_fp64(dev):
    G = load_golden(elbo_fixture.NAME)
    ph, g, ens = _mirrors(G, torch.double, dev)
    assert ens._weights() is not None and ens._inputs()[0].n_inputs == 256        # batched matrix-free update, pixel layout
    assert rel_err(ens.mean.cpu(), G['out_vo_mean']) < 1e-9
    assert rel_err(ens.logsigma.cpu(), G['out_vo_logsigma']) < 1e-8
    value, grads = elbo_fixture.run_elbo(g, ens, G, torch.double, dev)
    worst = elbo_fixture.compare_with_reference(value, grads, G, 1e-9)
    assert set(worst) >= {"g.logsigmas_y", "gp.fc.weight", "q_X.supervised.mean", "q_X.vo.logsigma", "f.fc.weight"}


def test_reference_elbo_on_the_mirrored_modules_fp32(dev):
    """The reference's model dtype (factories/model.py:181,224): float32 modules, the VO side stays double inside."""
    G = load_golden(elbo_fixture.NAME)
    ph, g, ens = _mirrors(G, torch.float32, dev)
    assert ens.mean.dtype == torch.float32
    value, grads = elbo_fixture.run_elbo(g, ens, G, torch.float32, dev)
    assert abs(value - float(G['out_elbo'])) < 2e-5 * abs(float(G['out_elbo']))
    for k, gr in grads.items():
        assert rel_err(gr, G['grad_' + k]) < 2e-3, k     # float32 sums over up to 1500 terms in the caller's torch ops


def test_fused_log_likelihood_matches_the_unfused_operator_path(dev):
    """ReducedOrderModelOperator.log_likelihood (fused epilogue, W u never written) == DiagonalGaussianLogLikelihood(Y,
    *g.forward(effprop, F)) of the drop-in path (utils.py:231-241 on components.py:296-298), value and gradients w.r.t.
    effprop, F and logsigmas_y; and against the oracle's restated ops on the CPU."""
    from oracle import elbo_ref, fem_p1, rom_ref
    G = load_golden(elbo_fixture.NAME)
    for dtype, tol in ((torch.double, 1e-10), (torch.float32, 2e-4)):
        ph, g, _ = _mirrors(G, dtype, dev)
        rng = np.random.RandomState(3)
        T = lambda a: torch.tensor(a, dtype=dtype, device=dev)
        Ns = G['in_sup_Y'].shape[0]
        with torch.no_grad():
            g.logsigmas_y.copy_(T(rng.normal(size=g.dim_out) * 0.2 - 1.0))
        outs = []
        for fused in (True, False):
            eff = T(G['init_q_X.supervised.mean']).requires_grad_(True)
            F = T(G['in_sup_F']).requires_grad_(True)
            g.logsigmas_y.grad = None
            if fused:
                L = g.log_likelihood(eff, F, T(G['in_sup_Y']))
            else:
                mu, ls = g(eff, F)
                L = elbo_ref.diagonal_gaussian_log_likelihood(T(G['in_sup_Y']), mu, 2 * ls)
            (3.0 * L).backward()
            outs.append((L.item(), eff.grad.clone(), F.grad.clone(), g.logsigmas_y.grad.clone()))
        assert abs(outs[0][0] - outs[1][0]) <= tol * abs(outs[1][0])
        for a, b in zip(outs[0][1:], outs[1][1:]):
            assert rel_err(a.cpu(), b.cpu()) < tol
        if dtype == torch.double:   # the oracle: the reference's torch ops on the CPU
            P = fem_p1.build_problem(int(G['nx']), int(G['nx']), int(G['refines']))
            eff = torch.tensor(G['init_q_X.supervised.mean'], requires_grad=True)
            ls = g.logsigmas_y.detach().cpu().clone().requires_grad_(True)
            mu = rom_ref.operator_forward_mean(torch.tensor(P['M']), torch.tensor(P['bc_dofs_rom']), torch.tensor(P['W']), eff,
                                               torch.tensor(G['in_sup_F']))
            L0 = elbo_ref.diagonal_gaussian_log_likelihood(torch.tensor(G['in_sup_Y']), mu, 2 * ls.repeat(Ns, 1))
            (3.0 * L0).backward()
            assert abs(outs[0][0] - L0.item()) <= 1e-10 * abs(L0.item())
            assert rel_err(outs[0][1].cpu(), eff.grad) < 1e-10 and rel_err(outs[0][3].cpu(), ls.grad) < 1e-10


def test_predictive_moments_match_their_definition_and_the_sampled_estimator(dev):
    """predictive_moments == W ubar / sqrt(W Cov W^T + sigma^2) computed with torch from the coarse solves (exact), and the
    reference's sampled estimator (propagate_samples + torch.mean / torch.std, generative.py:198-207) within Monte-Carlo
    error."""
    G = load_golden(elbo_fixture.NAME)
    ph, g, _ = _mirrors(G, torch.double, dev)
    rng = np.random.RandomState(5)
    N, S = 3, 256
    T = lambda a: torch.tensor(a, dtype=torch.double, device=dev)
    with torch.no_grad():
        g.logsigmas_y.copy_(T(rng.normal(size=g.dim_out) * 0.2 - 2.0))
    eff = T(G['init_q_X.vo.mean'][:N])[:, None, :] + 0.3 * T(rng.normal(size=(N, S, g.dim_in)))
    F = T(G['in_vo_F'][:N])
    y_mean, y_std = g.predictive_moments(eff, F)
    with torch.no_grad():
        u = g.rom.solve_log(eff.reshape(N * S, -1), F[:, None, :].expand(N, S, -1).reshape(N * S, -1)).reshape(N, S, -1)
        mu = torch.einsum('sk,nqk->nqs', g.W, u)                                   # [N,S,d]
        want_mean = mu.mean(dim=1)
        want_std = torch.sqrt(mu.var(dim=1, unbiased=True) + torch.exp(2 * g.logsigmas_y))
        assert rel_err(y_mean.cpu(), want_mean.cpu()) < 1e-11 and rel_err(y_std.cpu(), want_std.cpu()) < 1e-10
        # the reference's estimator: sample the output noise too (statistical agreement, S = 256)
        torch.manual_seed(0)
        ys = torch.stack([g.propagate_samples(eff[n], F[n].expand(S, -1)) for n in range(N)])
        assert (ys.mean(dim=1) - y_mean).abs().max() < 6 * (y_std / np.sqrt(S)).max()
        assert ((ys.std(dim=1) / y_std) - 1).abs().max() < 0.35

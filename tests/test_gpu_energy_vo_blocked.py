"""Blocked subspace-Newton step of the energy-type virtual observables for up to 256 weighting functions per data point
(csrc/vo_energy_blocked.cuh through gpde_vo_energy_step_blocked_f64) and the "blocked" route of
EnergyVirtualObservablesEnsemble.update:
    kernel     rho launch + energy_step_blocked, repeated  -> oracle/vo_ref.energy_vo_update per data point (1e-10),
               the one-launch kernel for m <= 64 (1e-12), the row split, determinism, the info word, argument errors
    ensemble   blocked route against the member loop (EnergyVirtualObservable.update per data point) on the same draws
"""
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


def _operands(plan, fom, gbc, rng, N, m, shared_V, shared_a, dev, n_steps=1):
    """Seeded inputs of an energy step: Gaussian V (M_n well conditioned for m <= d / 2), warm-started means and a
    different temperature per data point."""
    d = fom.dim_out
    T = lambda t: torch.tensor(t, device=dev)
    x = rng.normal(0.2, 0.6, size=(1 if shared_a else N, fom.dim_in))
    p = dict(x=x, g=rng.normal(size=(N, d)), prec=rng.uniform(0.5, 50.0, size=(N, d)), T_n=rng.uniform(0.05, 2.0, size=N),
             mean0=rng.normal(size=(N, d)),
             Vs=[rng.normal(size=(d, m)) if shared_V else rng.normal(size=(N, d, m)) for _ in range(n_steps)])
    p.update(a=torch.exp(T(x[0] if shared_a else x)), gbc_t=T(gbc), gt=T(p["g"]), pt=T(p["prec"]),
             it=T(1.0 / p["T_n"]), Vts=[T(V) for V in p["Vs"]])
    return p


def _steps(plan, p, step, info=None, mean=None, prec=None):
    """Newton steps (a rho launch, then ``step``) from the warm start; returns the updated means."""
    mean = torch.tensor(p["mean0"], device=p["gt"].device) if mean is None else mean
    for V in p["Vts"]:
        _, rho = plan.residual(p["a"], mean, p["gbc_t"], None, a_is_log=False)
        out = step(p["a"], V, rho, p["gt"], p["pt"] if prec is None else prec, p["it"], mean, info=info)
        assert out is mean
    return mean


# m in {1, 33, 64, 65, 100, 128, 129, 256} with m <= d / 2 (M_n is singular once m > d); d = 255 on 16 x 16, 1023 on
# 32 x 32, 4095 on 64 x 64
CASES = [(16, 16, m) for m in (1, 33, 64, 65, 100)] + [(32, 32, m) for m in (1, 33, 64, 65, 100, 128, 129, 256)] + \
        [(64, 64, 256)]


@pytest.mark.parametrize("nx,ny,m", CASES)
def test_energy_step_blocked_matches_oracle(nx, ny, m, dev):
    from oracle import vo_ref
    k = CASES.index((nx, ny, m))
    kind, shared_V, shared_a = ("ND", "NDP")[k % 2], bool(k % 3 == 0), bool(k % 4 == 1)
    N = 2 if nx == 64 else (1, 3, 5)[k % 3]
    plan, fom, asm, gbc, rng = _kernel_case(nx, ny, kind, N, 500 + k, dev)
    p = _operands(plan, fom, gbc, rng, N, m, shared_V, shared_a, dev, n_steps=3)
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    mean = _steps(plan, p, plan.energy_step_blocked, info=info)
    assert int(info.item()) == 0
    for n in range(N):
        K, f = asm.assemble(np.exp(p["x"][0 if shared_a else n]), gbc[n])
        want, _ = vo_ref.energy_vo_update(K, f, p["g"][n], p["prec"][n], p["mean0"][n],
                                          [V if shared_V else V[n] for V in p["Vs"]], p["T_n"][n])
        assert rel_err(mean[n].cpu(), want) < 1e-10, (n, rel_err(mean[n].cpu(), want))
    if m <= 64:        # the one-launch kernel on the same inputs
        mean1 = _steps(plan, p, plan.energy_step)
        assert rel_err(mean.cpu(), mean1.cpu()) < 1e-12


def test_energy_step_blocked_row_split_matches_unsplit_call(dev):
    """N = 1 at m = 256 splits the Gram pass over row segments; the same data point inside a batch of 64 runs unsplit."""
    plan, fom, asm, gbc, rng = _kernel_case(32, 32, "NDP", 64, 7, dev)
    m, N = 256, 64
    assert plan.posterior_blocked_workspace_bytes(1, m) > plan.posterior_blocked_workspace_bytes(N, m) // N
    p = _operands(plan, fom, gbc, rng, N, m, False, False, dev)
    mean = _steps(plan, p, plan.energy_step_blocked)
    for n in (0, 17):
        sl = slice(n, n + 1)
        q = dict(p, a=p["a"][sl], gbc_t=p["gbc_t"][sl], gt=p["gt"][sl], pt=p["pt"][sl], it=p["it"][sl],
                 mean0=p["mean0"][sl], Vts=[V[sl] for V in p["Vts"]])
        m1 = _steps(plan, q, plan.energy_step_blocked)
        assert rel_err(m1[0].cpu(), mean[n].cpu()) < 1e-13


@pytest.mark.parametrize("m", [100, 256])
def test_energy_step_blocked_is_deterministic(m, dev):
    plan, fom, asm, gbc, rng = _kernel_case(32, 32, "NDP", 6, 11, dev)
    N = 6
    p = _operands(plan, fom, gbc, rng, N, m, True, False, dev)
    mean = _steps(plan, p, plan.energy_step_blocked)
    for _ in range(3):
        assert torch.equal(_steps(plan, p, plan.energy_step_blocked), mean)
    perm = torch.tensor([3, 0, 5, 1, 4, 2], device=dev)
    q = dict(p, a=p["a"][perm], gbc_t=p["gbc_t"][perm], gt=p["gt"][perm], pt=p["pt"][perm], it=p["it"][perm],
             mean0=p["mean0"][perm.cpu().numpy()])
    assert torch.equal(_steps(plan, q, plan.energy_step_blocked), mean[perm])


def test_energy_step_blocked_indefinite_matrix_keeps_that_mean(dev):
    """prec = -1e6 on data point 1 makes its M indefinite: info word, its mean bitwise unchanged, and every other data
    point bitwise equal to a run (same N, so the same row split) in which data point 1 is a good one."""
    plan, fom, asm, gbc, rng = _kernel_case(32, 32, "NDP", 4, 13, dev)
    N, m = 4, 100
    p = _operands(plan, fom, gbc, rng, N, m, False, False, dev)
    prec_bad = p["pt"].clone()
    prec_bad[1] = -1e6
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    mean_bad = _steps(plan, p, plan.energy_step_blocked, info=info, prec=prec_bad)
    assert int(info.item()) == 2
    assert torch.equal(mean_bad[1], torch.tensor(p["mean0"][1], device=dev))
    info.zero_()
    mean_good = _steps(plan, p, plan.energy_step_blocked, info=info)
    assert int(info.item()) == 0
    keep = [0, 2, 3]
    assert torch.equal(mean_bad[keep], mean_good[keep]) and not torch.equal(mean_good[1], mean_bad[1])


def test_energy_step_blocked_errors(dev):
    from gpde_b200 import _lib
    plan, fom, asm, gbc, rng = _kernel_case(16, 16, "NDP", 3, 17, dev)
    N, m, d = 3, 100, fom.dim_out
    p = _operands(plan, fom, gbc, rng, N, m, True, False, dev)
    mean = torch.tensor(p["mean0"], device=dev)
    _, rho = plan.residual(p["a"], mean, p["gbc_t"], None, a_is_log=False)
    args = (rho, p["gt"], p["pt"], p["it"], mean)
    V = p["Vts"][0]
    with pytest.raises(RuntimeError):                                        # m = 257: GPDE_ERR_SIZE
        plan.energy_step_blocked(p["a"], torch.zeros(d, 257, dtype=torch.float64, device=dev), *args)
    lib, P = plan._lib, lambda t: _lib.ptr(t, dev)
    need = plan.posterior_blocked_workspace_bytes(N, m)
    ws = torch.zeros(need + 64, dtype=torch.uint8, device=dev)
    st = _lib.stream_of(dev)
    before = mean.clone()

    def call(mm=m, a_stride=plan.n_inputs, v_stride=0, wsp=P(ws), nbytes=need, n=N):
        return lib.gpde_vo_energy_step_blocked_f64(plan.handle, P(p["a"]), a_stride, P(V), v_stride, mm, P(rho), P(p["gt"]),
                                                   P(p["pt"]), P(p["it"]), P(mean), None, wsp, nbytes, n, st)
    assert call(mm=0) == -1                                                   # GPDE_ERR_ARG
    assert call(mm=257, nbytes=ws.numel()) == -3                              # GPDE_ERR_SIZE
    assert call(v_stride=d * m + 1) == -1
    assert call(a_stride=plan.n_inputs + 1) == -1
    assert call(wsp=None) == -1                                               # null workspace
    assert call(wsp=ctypes.c_void_p(ws.data_ptr() + 8)) == -1                 # misaligned
    assert call(nbytes=need - 1) == -1                                        # one byte short
    assert call(n=0, wsp=None, nbytes=0) == 0                                 # N = 0: nothing to do
    torch.cuda.synchronize()
    assert torch.equal(mean, before)
    with pytest.raises(ValueError):                                           # per-data-point V of another batch size
        plan.energy_step_blocked(p["a"], V.expand(N + 1, d, m).contiguous(), *args)
    assert call() == 0
    torch.cuda.synchronize()
    assert torch.isfinite(mean).all() and not torch.equal(mean, before)


# ------------------------------------------------------------------------------------------------ ensemble
def _ensemble(dev, N=5, n_it=3, sampler=None, seed=4):
    """32 x 32 fine mesh (d = 1023), NDP boundary values, one sampler shared by the data points."""
    from gpde_b200 import VirtualObservables as VO
    from gpde_b200.physics import setup_physics, BoundaryConditionEnsemble
    rng = np.random.RandomState(seed)
    ph = setup_physics(4, 4, 3, "NDP")
    fom = ph['fom']
    bce = BoundaryConditionEnsemble(ph, N, "NDP", rng=rng)
    qpe = VO.QuerryPointEnsemble.FromArrays(rng.normal(0.0, 0.5, size=(N, fom.dim_in)), bce, fom, device=dev)
    ens = VO.EnergyVirtualObservablesEnsemble(qpe, n_it, sampler(qpe), torch.double, dev)
    ens.set_linear_temperature_schedule(T_init=1.0, T_final=1e-2, num_steps=4)
    return ens, fom


def _inputs(fom, N, seed):
    rng = np.random.RandomState(seed)
    return [(rng.normal(size=(N, fom.dim_out)), rng.uniform(1.0, 30.0, size=(N, fom.dim_out))) for _ in range(3)]


def _run(ens, inputs, dev):
    out = []
    for it, (G, P) in enumerate(inputs):
        ens.update(torch.tensor(G, device=dev), torch.tensor(P, device=dev), it)
        out.append((ens.mean.clone(), ens.vars.clone(), [vo.temperature for vo in ens]))
    return out


def _assert_same(out_a, out_b, tol=1e-10):
    for (ma, va, ta), (mb, vb, tb) in zip(out_a, out_b):
        assert rel_err(ma.cpu(), mb.cpu()) < tol
        assert torch.equal(va, vb)
        assert ta == tb


def _sketch(m):
    from gpde_b200 import VirtualObservables as VO
    return lambda qpe: VO.GaussianSketchingSampler(qpe[0], m)


@pytest.mark.parametrize("m,n_it", [(65, 1), (65, 3), (128, 1), (128, 3)])
def test_blocked_route_matches_member_loop(m, n_it, dev):
    outs = []
    for route in ("blocked", "members", "chunked"):
        ens, fom = _ensemble(dev, n_it=n_it, sampler=_sketch(m))
        ens.max_blocked_m = 256
        ens.batched_update = route != "members"
        if route == "chunked":
            ens.max_stack_bytes = 1                                          # one data point per chunk
        np.random.seed(21)
        outs.append(_run(ens, _inputs(fom, ens.N, 3), dev))
        assert ens.last_update_route == ("members" if route == "members" else "blocked")
    _assert_same(outs[0], outs[1])
    _assert_same(outs[0], outs[2], tol=1e-12)


def test_blocked_route_with_m_found_in_the_draws(dev):
    """A sampler without an ``m`` attribute (m = 70): the blocked route on the draws already made, in member-loop order."""
    from gpde_b200 import VirtualObservables as VO

    class Recording(VO.BaseSampler):
        """Draw k is a seeded matrix whose first entry is k: the record shows which draw went where."""

        def __init__(self, qp):
            super().__init__(qp)
            self.rng, self.calls = np.random.RandomState(12), 0

        def _sample(self):
            V = self.rng.normal(size=(self.qp.dim_out, 70))
            V[0, 0] = self.calls
            self.calls += 1
            return V

    outs = []
    for batched in (True, False):
        ens, fom = _ensemble(dev, n_it=2, sampler=lambda qpe: Recording(qpe[0]))
        ens.max_blocked_m = 256
        ens.batched_update = batched
        outs.append(_run(ens, _inputs(fom, ens.N, 6), dev))
        assert ens.last_update_route == ("blocked" if batched else "members")
        assert ens[0]._sampler.calls == 3 * 2 * ens.N
        assert all(isinstance(vo._sampler, Recording) for vo in ens)          # the members' samplers are restored
    _assert_same(*outs)


def test_member_loop_above_the_blocked_limit(dev):
    # under the defaults the blocked route is off: m = 70 takes the member loop
    ens, fom = _ensemble(dev, n_it=1, sampler=_sketch(70))
    assert ens.max_blocked_m == 64
    inputs = _inputs(fom, ens.N, 6)[:1]
    _run(ens, inputs, dev)
    assert ens.last_update_route == "members"
    # m = 257 is above max_blocked_m = 256
    ens, fom = _ensemble(dev, n_it=1, sampler=_sketch(257))
    ens.max_blocked_m = 256
    _run(ens, inputs, dev)
    assert ens.last_update_route == "members"


# one blocked ensemble update (n_it = 2) under torch.profiler; prints its route and the names of its device kernels
_PROFILE_SCRIPT = """
import json, sys
sys.path.insert(0, sys.argv[1])
import numpy as np, torch
import test_gpu_energy_vo_blocked as t
dev = torch.device("cuda", 0)
ens, fom = t._ensemble(dev, n_it=2, sampler=t._sketch(128))
ens.max_blocked_m = 256
inputs = t._inputs(fom, ens.N, 8)
t._run(ens, inputs[:1], dev)
G, P = (torch.tensor(x, device=dev) for x in inputs[1])
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    ens.update(G, P, 1)
    torch.cuda.synchronize()
names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
print(json.dumps({"route": ens.last_update_route, "names": names}))
"""


def test_blocked_route_runs_only_project_kernels(dev):
    """The capture runs in a process of its own, so that this process's profiler state stays as the other tests find it."""
    import json
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    res = subprocess.run([sys.executable, "-s", "-c", _PROFILE_SCRIPT, here], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-4000:]
    out = json.loads(res.stdout.strip().splitlines()[-1])
    assert out["route"] == "blocked"
    names = out["names"]
    for k in ("vo_energy_gram_kernel", "vo_post_factor_kernel", "vo_energy_apply_kernel"):
        assert sum(k in s for s in names) == 2, k                             # one per Newton iteration
    vendor = ("cublas", "cusolver", "potrf", "trsm", "syrk", "gemm", "getrf", "xmma", "cutlass", "magma")
    assert not [s for s in names if "gpde" not in s and any(v in s.lower() for v in vendor)]

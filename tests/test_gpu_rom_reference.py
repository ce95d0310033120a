"""Every route of the coarse-grained-model kernels (csrc/rom.cu, rom_tps.cuh, rom_tpw.cuh) against the refined float64
reference of oracle.rom_ref.rom_reference, entry by entry: |out - ref| <= c eps64 S with the per-entry rounding-error
scale S and c = 4 (hbw + T + 4) (float32 outputs are allowed their own rounding on top).  Routes: thread per sample
(lanes 1), windowed thread per sample (lanes 2), cooperative (lanes 8 / 16 / 32), on meshes, diagonals, rectangles and
Dirichlet sets beyond the ones each kernel was written for."""
import zlib

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import rom_ref

pytestmark = pytest.mark.gpu

REACHED = set()      # (lanes, dtype) of every case run, for the coverage test at the end


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


class _Phys(object):
    def __init__(self, bc, free):
        self.constrained_dofs, self.free_dofs = np.asarray(bc), np.asarray(free)


def _mesh(nx, ny, diagonal="right", Lx=1.0, Ly=1.0, bc=None):
    from oracle import fem_p1
    c, cells = fem_p1.unit_square_mesh(nx, ny, diagonal)
    c = c * np.array([Lx, Ly])
    M = fem_p1.rom_element_tensor(c, cells)
    if bc is None:      # left-right Dirichlet
        bc = [i for i, (x, _) in enumerate(c) if abs(x) < 1e-12 or abs(x - Lx) < 1e-12]
    bc = np.array(sorted(bc), dtype=np.int64)
    free = np.array(sorted(set(range(len(c))) - set(bc.tolist())), dtype=np.int64)
    return M, bc, free


def _rom(M, bc, free, dtype, dev, monkeypatch=None, coop=False):
    from gpde_b200.ROM import ROM
    if monkeypatch is not None:
        if coop:
            monkeypatch.setenv("GPDE_ROM_PATH", "coop")
        else:
            monkeypatch.delenv("GPDE_ROM_PATH", raising=False)
    # M stays float64 for float32 I/O too (the plan converts it to float64): the kernels then solve exactly the system
    # of the reference; a float32-rounded M on non-square cells breaks the zero row sums of the element matrices
    rom = ROM(_Phys(bc, free), torch.tensor(M, dtype=torch.float64, device=dev), dtype, dev)
    rom._get_plan()      # the path is read here
    if monkeypatch is not None:
        monkeypatch.delenv("GPDE_ROM_PATH", raising=False)
    return rom


# name -> (mesh arguments, lanes of the route, force the cooperative kernels)
_8x8_COLS = [i for i in range(81) if i % 9 in (0, 4)]
CASES = {
    "4x4": (dict(nx=4, ny=4), 1, False),
    "4x4-left": (dict(nx=4, ny=4, diagonal="left"), 1, False),
    "4x4-rect": (dict(nx=4, ny=4, Lx=2.0, Ly=0.5), 1, False),
    "4x4-bcA": (dict(nx=4, ny=4, bc=[0, 1, 3, 4, 8, 9, 13, 14, 18, 19]), 1, False),
    "4x4-bcB": (dict(nx=4, ny=4, bc=[2, 3, 7, 8, 12, 13, 17, 18, 22, 23]), 1, False),
    "4x4-bcC": (dict(nx=4, ny=4, bc=[5, 6, 10, 11, 15, 16, 20, 21, 23, 24]), 1, False),
    "8x8": (dict(nx=8, ny=8), 2, False),
    "8x8-left": (dict(nx=8, ny=8, diagonal="left"), 2, False),
    "8x8-rect": (dict(nx=8, ny=8, Lx=2.0, Ly=0.5), 2, False),
    "8x8-cols04": (dict(nx=8, ny=8, bc=_8x8_COLS), 2, False),
    # the alternating diagonal gives 8 terms on some diagonal entries (tps holds 6) and couplings inside the band (tpw)
    "4x4-alternating": (dict(nx=4, ny=4, diagonal="alternating"), 8, False),
    # n_free = 15 and hbw = 3, but a free dof between two Dirichlet dofs has 4 right-hand-side terms (tps holds 2)
    "4x4-bc-issue": (dict(nx=4, ny=4, bc=[4, 5, 8, 9, 10, 15, 16, 19, 20, 24]), 8, False),
    "2x2": (dict(nx=2, ny=2), 8, False),
    "3x9": (dict(nx=3, ny=9), 8, False),
    "4x4-coop": (dict(nx=4, ny=4), 8, True),
    "2x72": (dict(nx=2, ny=72), 8, False),
    "5x5": (dict(nx=5, ny=5), 16, False),
    "6x3": (dict(nx=6, ny=3), 16, False),
    "12x12": (dict(nx=12, ny=12), 32, False),
    "16x9": (dict(nx=16, ny=9), 32, False),
    "12x1": (dict(nx=12, ny=1), 32, False),
    "8x8-coop": (dict(nx=8, ny=8), 32, True),
    "8x8-alternating": (dict(nx=8, ny=8, diagonal="alternating"), 32, False),
    # widest band the plan accepts under the 290-cell cap: hbw 50 (52x1, hbw 51, exceeds 227 KB per CTA)
    "51x1": (dict(nx=51, ny=1), 32, False),
}


def _inputs(M, bc, B, rng, dtype):
    """logX rows: N(0.4, 0.8), then U[-12, 12] (high contrast), then the libm branch of exp (|X| > 700): columns at -705,
    -750 and -inf, and (float64) a sample with every entry at 705 + N(0, 0.5).  Where a diagonal coefficient of M
    exceeds 4 (skinny elements) that sample is lowered by its log so that K and the bounds stay finite, but not below
    700.2.  Non-zero free loads, random gbar everywhere."""
    n, _, E = M.shape
    top = max(705.0 - max(0.0, np.log(np.abs(M).sum(axis=2).diagonal().max() / 4.0)), 701.5)
    logX = rng.normal(0.4, 0.8, size=(B, E))
    logX[B // 3: 2 * B // 3] = rng.uniform(-12, 12, size=(2 * B // 3 - B // 3, E))
    if B >= 4:
        logX[-3, ::5] = -705.0
        logX[-3, 1::7] = -750.0
        logX[-2, 2::6] = -np.inf
        if dtype == torch.float64:
            logX[-1] = np.maximum(top + rng.normal(0, 0.5, size=E), 700.2)
    F = rng.normal(size=(B, n)) * 0.3
    F[:, bc] = rng.uniform(-0.5, 0.5, size=(B, len(bc)))
    gbar = rng.normal(size=(B, n))
    t = lambda a: torch.tensor(a, dtype=dtype)
    return t(logX), t(F), t(gbar)


def _check(name, out, ref, S, c, fp32, ratios):
    r = rom_ref.bound_ratio(out, ref, S, fp32=fp32)
    ratios[name] = max(ratios.get(name, 0.0), r)
    assert r <= c, (name, r, c)


def _run_case(rom, M, bc, dtype, dev, Xh, Fh, gbh, x_is_log, ratios):
    """Forward with and without a factor, adjoint with the stash, without it and without gradF, and the autograd
    surface, each against the reference of the inputs it was given."""
    from gpde_b200 import ROM as rom_mod
    plan = rom._get_plan()
    fp32 = dtype == torch.float32
    X, F, gb = Xh.to(dev), Fh.to(dev), gbh.to(dev)
    ref = rom_ref.rom_reference(M, bc, Xh.double().numpy(), Fh.double().numpy(), gbh.double().numpy(), x_is_log)
    c = ref["c"]
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    u, factor = rom_mod._launch_forward(plan, X, F, x_is_log, want_factor=True, info=info)
    u2, _ = rom_mod._launch_forward(plan, X, F, x_is_log, want_factor=False, info=info)
    assert int(info.item()) == 0
    for uu in (u, u2):
        uc = uu.cpu()
        _check("u", uc.double().numpy(), ref["u"], ref["S_u"], c, fp32, ratios)
        assert torch.equal(uc[:, bc], Fh[:, bc])          # Dirichlet values: exact
    # the adjoint against the reference of the u it is given
    refa = ref if not fp32 else rom_ref.rom_reference(M, bc, Xh.double().numpy(), Fh.double().numpy(),
                                                      gbh.double().numpy(), x_is_log, u=u.cpu().double().numpy())
    variants = [(factor, True), (None, True), (factor, False)]
    for fac, want_gF in variants:
        gX, gF = rom_mod._launch_adjoint(plan, X, u, fac, gb, x_is_log, want_gradF=want_gF)
        _check("gX", gX.cpu().double().numpy(), refa["gX"], refa["S_gX"], c, fp32, ratios)
        if want_gF:
            _check("gF", gF.cpu().double().numpy(), refa["lam"], refa["S_lam"], c, fp32, ratios)
    # autograd surface: the whole chain (float64: against the exact u; float32: against the u of the forward)
    Xg = X.clone().requires_grad_(True)
    Fg = F.clone().requires_grad_(True)
    ua = rom.solve_log(Xg, Fg) if x_is_log else rom(Xg, Fg)
    ua.backward(gb)
    assert torch.equal(ua.detach(), u)
    _check("gX", Xg.grad.cpu().double().numpy(), refa["gX"], refa["S_gX"], c, fp32, ratios)
    _check("gF", Fg.grad.cpu().double().numpy(), refa["lam"], refa["S_lam"], c, fp32, ratios)
    return ref


RATIOS = {}


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("case", list(CASES))
def test_route_against_refined_reference(case, dtype, dev, monkeypatch):
    margs, lanes, coop = CASES[case]
    M, bc, free = _mesh(**margs)
    rom = _rom(M, bc, free, dtype, dev, monkeypatch, coop)
    plan = rom._get_plan()
    assert plan.lanes == lanes, (case, plan.lanes)
    REACHED.add((lanes, dtype))
    rng = np.random.RandomState(zlib.crc32(case.encode()))
    B = 300 if M.shape[0] <= 100 else 129
    X, F, gb = _inputs(M, bc, B, rng, dtype)
    ratios = {}
    _run_case(rom, M, bc, dtype, dev, X, F, gb, True, ratios)
    # conductivity input (the 705 row would overflow float32: clipped there)
    xc = torch.exp(X.double().clamp(-700.0, 700.0 if dtype == torch.float64 else 80.0)) + 1e-8
    _run_case(rom, M, bc, dtype, dev, xc.to(dtype), F, gb, False, ratios)
    RATIOS[(case, lanes, str(dtype))] = ratios
    print("ratios", case, lanes, dtype, {k: round(v, 2) for k, v in ratios.items()})


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("case", ["4x4", "8x8", "2x2", "5x5", "12x12", "8x8-coop"])
def test_batch_edges_and_ragged_tail(case, dtype, dev, monkeypatch):
    """B = 0, 1, one below and one above the CTA granularity (128 samples for tps / tpw, 128 / G for the cooperative
    kernels), and a ragged tail whose last sample alone is bad (flag raised, every other sample still right)."""
    margs, lanes, coop = CASES[case]
    M, bc, free = _mesh(**margs)
    rom = _rom(M, bc, free, dtype, dev, monkeypatch, coop)
    assert rom._get_plan().lanes == lanes
    gran = 128 if lanes <= 2 else 128 // lanes
    rng = np.random.RandomState(7)
    for B in sorted({0, 1, gran - 1, gran + 1, 2 * gran + 3}):
        X, F, gb = _inputs(M, bc, B, rng, dtype)
        X[:] = X.clamp(-3, 3)
        ratios = {}
        _run_case(rom, M, bc, dtype, dev, X, F, gb, True, ratios)
    # ragged tail: the last sample holds a non-positive conductivity
    B = 2 * gran + 3
    X, F, gb = _inputs(M, bc, B, rng, dtype)
    x = torch.exp(X.double().clamp(-3, 3)).to(dtype)
    x[-1, -1] = 0.0
    xd = x.to(dev)
    rom.deferred_checks = True
    u = rom(xd, F.to(dev))
    with pytest.raises(ValueError):
        rom.check()
    ref = rom_ref.rom_reference(M, bc, x[:-1].double().numpy(), F[:-1].double().numpy(), gb[:-1].double().numpy(), False)
    assert rom_ref.bound_ratio(u[:-1].cpu().double().numpy(), ref["u"], ref["S_u"],
                               fp32=dtype == torch.float32) <= ref["c"]


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("case", ["4x4", "8x8", "5x5", "12x12", "4x4-coop", "8x8-coop"])
def test_info_word_threshold_nan_and_not_spd(case, dtype, dev, monkeypatch):
    """Bit 1: x <= 1e-12 (the next double above does not flag; in float32 float(1e-12) flags and 2e-12 does not), NaN.
    Bit 2: M -> -M makes every pivot negative; ROM.check raises RuntimeError, ValueError when bit 1 is also set."""
    margs, lanes, coop = CASES[case]
    M, bc, free = _mesh(**margs)
    E, n = M.shape[2], M.shape[0]
    rom = _rom(M, bc, free, dtype, dev, monkeypatch, coop)
    assert rom._get_plan().lanes == lanes
    F = torch.zeros(5, n, dtype=dtype, device=dev)

    def flag(v, r=rom):
        X = torch.ones(5, E, dtype=torch.float64)
        X[3, E // 2] = v
        r(X.to(dtype).to(dev), F)
        return int(r._info.item())

    rom.deferred_checks = True
    lo, hi = (1e-12, np.nextafter(1e-12, 1.0)) if dtype == torch.float64 else (float(np.float32(1e-12)), 2e-12)
    assert flag(lo) & 1
    rom._info.zero_()
    assert flag(hi) == 0
    assert flag(float("nan")) & 1
    rom._info.zero_()
    neg = _rom(-M, bc, free, dtype, dev, monkeypatch, coop)
    assert neg._get_plan().lanes == lanes
    neg.deferred_checks = True
    assert flag(1.0, neg) == 2
    with pytest.raises(RuntimeError):
        neg.check()
    assert flag(0.0, neg) == 3
    with pytest.raises(ValueError):
        neg.check()


def test_plans_the_library_refuses(dev):
    """No free dofs (1x12), and meshes under the 290-cell cap whose cooperative kernels need more than 227 KB of shared
    memory per CTA (36x4, and 52x1 just past the widest accepted band): refused when the plan is created."""
    from gpde_b200 import _lib
    from gpde_b200.ROM import ROM
    for nx, ny in ((1, 12), (36, 4), (52, 1)):
        M, bc, free = _mesh(nx, ny)
        assert M.shape[2] <= 290
        rom = ROM(_Phys(bc, free), torch.tensor(M, device=dev), torch.float64, dev)
        with pytest.raises(_lib.GpdeLibraryError):
            rom._get_plan()
    M, bc, free = _mesh(51, 1)
    plan = ROM(_Phys(bc, free), torch.tensor(M, device=dev), torch.float64, dev)._get_plan()
    assert plan.half_bandwidth == 50 and plan.lanes == 32


@pytest.mark.parametrize("case", ["4x4", "8x8", "5x5"])
def test_unsorted_and_duplicated_dirichlet_list(case, dev):
    margs, lanes, _ = CASES[case]
    M, bc, free = _mesh(**margs)
    rng = np.random.RandomState(2)
    messy = np.concatenate([rng.permutation(bc), bc[:3]])
    X, F, gb = _inputs(M, bc, 77, rng, torch.float64)
    out = []
    for b in (bc, messy):
        rom = _rom(M, b, free, torch.float64, dev)
        assert rom._get_plan().lanes == lanes
        Xg = X.to(dev).requires_grad_(True)
        Fg = F.to(dev).requires_grad_(True)
        u = rom.solve_log(Xg, Fg)
        u.backward(gb.to(dev))
        out.append((u.detach(), Xg.grad, Fg.grad))
    for a, b in zip(*out):
        assert torch.equal(a, b)


@pytest.mark.parametrize("case", ["4x4", "8x8", "4x4-rect", "8x8-alternating"])
@pytest.mark.parametrize("dirichlet", [True, False])
def test_get_stiffness_is_exact_on_dyadic_inputs(case, dirichlet, dev):
    """Dyadic conductivities k/64 on meshes whose element tensors are dyadic: M x is exact in float64, so GetStiffness must
    equal it bitwise.  The batch makes n^2 B exceed the grid of min(want, 16 SMs) CTAs of 256 threads (grid-stride loop)."""
    from gpde_b200.ROM import ROM
    margs, _, _ = CASES[case]
    M, bc, free = _mesh(**margs)
    n, E = M.shape[0], M.shape[2]
    assert np.array_equal(M * 2.0 ** 20, np.round(M * 2.0 ** 20))      # dyadic entries
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    B = (16 * sms * 256) // (n * n) + 7
    assert n * n * B > 16 * sms * 256
    rng = np.random.RandomState(5)
    x = rng.randint(1, 64 * 8, size=(B, E)) / 64.0
    want = np.einsum('ije,be->ijb', M, x)
    if dirichlet:
        want[bc] = 0.0
        want[bc, bc] = 1.0
    rom = ROM(_Phys(bc, free), torch.tensor(M, device=dev), torch.float64, dev)
    K = rom.GetStiffness(torch.tensor(x, device=dev), DirichletBC=dirichlet)
    assert torch.equal(K.cpu(), torch.tensor(want))


@pytest.mark.parametrize("case", ["4x4", "8x8", "5x5"])
def test_per_entry_check_catches_what_the_global_measure_misses(case, dev):
    """A plan built from M' whose one edge weight of one element differs by delta = 1e-11 relative (kept symmetric with
    zero row sums: the same route is taken) against the reference of M: the old max|a-b|/max|b| < 1e-10 passes, the
    per-entry check fails on u and on dL/dX."""
    from gpde_b200 import ROM as rom_mod
    margs, lanes, _ = CASES[case]
    M, bc, free = _mesh(**margs)
    fr = set(free.tolist())
    e, a, b = next((e, int(a), int(b)) for e in range(M.shape[2] // 2, M.shape[2]) for a, b in zip(*np.nonzero(M[:, :, e]))
                   if a < b and a in fr and b in fr)     # an edge between two free dofs
    Mp = M.copy()
    d = 1e-11 * M[a, b, e]
    Mp[a, b, e] += d; Mp[b, a, e] += d; Mp[a, a, e] -= d; Mp[b, b, e] -= d
    rom = _rom(Mp, bc, free, torch.float64, dev)
    plan = rom._get_plan()
    assert plan.lanes == lanes
    rng = np.random.RandomState(11)
    X, F, gb = _inputs(M, bc, 64, rng, torch.float64)
    X = X.clamp(-2, 2)
    Xd, Fd, gd = X.to(dev), F.to(dev), gb.to(dev)
    u, factor = rom_mod._launch_forward(plan, Xd, Fd, True, want_factor=True)
    gX, _ = rom_mod._launch_adjoint(plan, Xd, u, factor, gd, True)
    ref = rom_ref.rom_reference(M, bc, X.numpy(), F.numpy(), gb.numpy(), True)
    u, gX = u.cpu().numpy(), gX.cpu().numpy()
    assert rel_err(u, ref["u"]) < 1e-10 and rel_err(gX, ref["gX"]) < 1e-10
    assert rom_ref.bound_ratio(u, ref["u"], ref["S_u"]) > ref["c"]
    assert rom_ref.bound_ratio(gX, ref["gX"], ref["S_gX"]) > ref["c"]


def test_every_route_reached_in_both_dtypes():
    """Runs after the route tests (file order): lanes 1, 2, 8, 16 and 32 in float64 and float32."""
    if not REACHED:
        pytest.skip("route tests not run")
    want = {(l, d) for l in (1, 2, 8, 16, 32) for d in (torch.float64, torch.float32)}
    assert want <= REACHED, sorted(want - REACHED, key=str)
    for k in sorted(RATIOS, key=str):
        print("max err / (eps S)", k, {n: round(v, 2) for n, v in RATIOS[k].items()})

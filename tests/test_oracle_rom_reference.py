"""CPU check of oracle.rom_ref.rom_reference (the refined reference and per-entry bounds the GPU tests of the
coarse-grained-model kernels use) against the closed-form and autograd restatements of the same model."""
import numpy as np
import pytest
import torch

from oracle import fem_p1, rom_ref


def _problem(nx, ny, B, seed, diagonal="right"):
    rng = np.random.RandomState(seed)
    c, cells = fem_p1.unit_square_mesh(nx, ny, diagonal)
    M = fem_p1.rom_element_tensor(c, cells)
    bc, _, free = fem_p1.dirichlet_left_right(c, "ND")
    F = rng.normal(size=(B, len(c)))
    logX = rng.normal(0.4, 0.8, size=(B, len(cells)))
    gbar = rng.normal(size=(B, len(c)))
    return M, bc, free, logX, F, gbar


@pytest.mark.parametrize("nx,ny,diagonal", [(2, 2, "right"), (4, 4, "right"), (3, 5, "alternating"), (4, 4, "left")])
def test_reference_matches_closed_form_and_autograd(nx, ny, diagonal):
    M, bc, free, logX, F, gbar = _problem(nx, ny, 7, nx * 10 + ny, diagonal)
    ref = rom_ref.rom_reference(M, bc, logX, F, gbar, x_is_log=True)
    u0, gX0, gF0 = rom_ref.rom_fwd_adjoint_closed_form(M, bc, free, logX, F, gbar)
    u1, gX1, gF1 = rom_ref.rom_fwd_adjoint(torch.tensor(M), torch.tensor(bc), torch.tensor(logX), torch.tensor(F),
                                           torch.tensor(gbar))
    for a, b in ((ref["u"], u0), (ref["gX"], gX0), (ref["lam"], gF0), (ref["u"], u1.numpy()), (ref["gX"], gX1.numpy()),
                 (ref["lam"], gF1.numpy())):
        assert np.abs(a - b).max() <= 1e-12 * np.abs(b).max()
    assert np.array_equal(ref["u"][:, bc], F[:, bc])
    # the refined residuals are at the extended precision's level, far below float64's
    assert ref["res_u"] < 1e-17 and ref["res_lam"] < 1e-17
    # conductivity input gives the same u; its gradient lacks the chain-rule factor exp(X)
    x = np.exp(logX) + 1e-8
    refx = rom_ref.rom_reference(M, bc, x, F, gbar, x_is_log=False)
    assert np.abs(refx["u"] - ref["u"]).max() <= 1e-13 * np.abs(ref["u"]).max()
    assert np.abs(refx["gX"] * np.exp(logX) - ref["gX"]).max() <= 1e-13 * np.abs(ref["gX"]).max()


def test_bound_ratio_and_scales():
    M, bc, free, logX, F, gbar = _problem(4, 4, 5, 3)
    ref = rom_ref.rom_reference(M, bc, logX, F, gbar, x_is_log=True)
    assert ref["hbw"] == 3 and ref["T"] == 6 and ref["c"] == 4 * (3 + 6 + 4)
    # scales are at least the magnitude of what they bound (|K^-1||K||u| >= |u|); exact entries have scale 0
    assert np.all(ref["S_u"][:, free] >= np.abs(ref["u"][:, free]) * (1 - 1e-12))
    assert np.all(ref["S_u"][:, bc] == 0)
    assert np.all(ref["S_lam"] >= np.abs(ref["lam"]) * (1 - 1e-12))
    assert rom_ref.bound_ratio(ref["u"], ref["u"], ref["S_u"]) == 0.0
    # one rounding unit of S is ratio 1; a float32 rounding of the output is forgiven only in float32 mode
    u = ref["u"] + rom_ref.EPS64 * ref["S_u"]
    assert 0.5 < rom_ref.bound_ratio(u, ref["u"], ref["S_u"]) < 2.0   # (the sum itself rounds)
    u32 = ref["u"].astype(np.float32)
    assert rom_ref.bound_ratio(u32, ref["u"], ref["S_u"], fp32=True) == 0.0
    assert rom_ref.bound_ratio(u32, ref["u"], ref["S_u"]) > 1e6
    # a given u enters the gradient as an exact input
    refg = rom_ref.rom_reference(M, bc, logX, F, gbar, x_is_log=True, u=u32.astype(np.float64))
    _, gX0, _ = rom_ref.rom_fwd_adjoint_closed_form(M, bc, free, logX, F, gbar)
    lam_f = refg["lam"].copy(); lam_f[:, bc] = 0
    want = -np.einsum('bi,ije,bj->be', lam_f, M, u32.astype(np.float64)) * np.exp(logX)
    assert np.abs(refg["gX"] - want).max() <= 1e-13 * np.abs(want).max()
    assert np.abs(refg["gX"] - gX0).max() > 1e-9 * np.abs(gX0).max()


def test_empty_batch():
    M, bc, free, logX, F, gbar = _problem(2, 2, 0, 1)
    ref = rom_ref.rom_reference(M, bc, logX, F, gbar, x_is_log=True)
    assert ref["u"].shape == (0, 9) and ref["gX"].shape == (0, 8)
    assert rom_ref.bound_ratio(ref["u"], ref["u"], ref["S_u"]) == 0.0

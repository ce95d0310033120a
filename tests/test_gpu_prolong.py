"""The prolongation kernels of csrc/prolong.cu against a float64 reference with a dense W on the CPU: y = W u and its
transpose, the fused Gaussian log-likelihood epilogue and the Monte-Carlo predictive moments, in FP64 and FP32 I/O.

The reference follows include/gpde_b200.h: y = u W^T, gu = gy W; e = (Y - u W^T) exp(-ls),
L_b = -1/2 sum_i (2 ls_i + e_bi^2 + log 2 pi), gu = (e exp(-ls)) W, gls_i = sum_b (e_bi^2 - 1); ubar / C the two-pass sample
mean / unbiased covariance of u[n,:,:], y_mean = W ubar, y_std = sqrt(diag(W C W^T) + exp(2 ls)).  FP32 cases apply it to the
float-rounded inputs, and W always comes from the float64 array the plan was built from.

Errors are measured per row (max_b max_i |a - ref| / max_i |ref_b|), so that one wrong small row of a batch of large ones
cannot hide.  FP32 calls do their arithmetic in double: double outputs (L, gls) are held to the FP64 tolerances, float
outputs to 4 float ulps of the row maximum."""
import functools
import math

import numpy as np
import pytest
import scipy.sparse
import torch

pytestmark = pytest.mark.gpu

LOG2PI = math.log(2.0 * math.pi)
DTYPES = [torch.float64, torch.float32]
# (nx_rom, num_refines): 16x16, 32x32 (cfg 1 and 5), 64x64 (cfg 2) fine meshes on the 4x4 coarse mesh, 128x128 (cfg 3) on 8x8
MESHES = {"16x16": (4, 2), "32x32": (4, 3), "64x64": (4, 4), "128x128": (8, 4)}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


@functools.lru_cache(maxsize=None)
def _physics(nx, refines):
    from gpde_b200.physics import setup_physics
    return setup_physics(nx, nx, refines, "ND")


def _synthetic_W(d, n, seed):
    """Sparse W with dyadic entries that P1 never produces: row 5 empty, column 7 empty, row 10 with 9 non-zeros and
    column 3 with 100 (the lane loops of the column kernels wrap three times)."""
    rng = np.random.RandomState(seed)
    W = np.zeros((d, n))
    for i in range(d):
        cols = rng.choice(n, size=rng.randint(1, 4), replace=False)
        W[i, cols] = rng.randint(1, 16, size=cols.size) / 16.0
    W[10, rng.choice(n, size=9, replace=False)] = rng.randint(-15, 16, size=9) / 16.0 + 1.0 / 32
    W[rng.choice(np.arange(11, d), size=100, replace=False), 3] = rng.randint(1, 16, size=100) / 16.0
    W[5, :] = 0.0
    W[:, 7] = 0.0
    assert (W[10] != 0).sum() > 3 and (W[:, 3] != 0).sum() > 32
    return W


def _W(mesh):
    if mesh == "synthetic":
        return _synthetic_W(300, 40, 11)
    return _physics(*MESHES[mesh])["W"]


def _plan(W, dev):
    from gpde_b200.components import _ProlongPlan
    return _ProlongPlan(torch.tensor(W, dtype=torch.float64), dev)


def _dyadic(rng, shape, scale=1.0):
    """Values with 16 fractional bits: exact in float32, and every product with the (dyadic) entries of W and every sum
    of a row's three products is exact in double -- W u of the reference carries no rounding of its own."""
    return np.round(rng.normal(size=shape) * scale * 2.0 ** 16) / 2.0 ** 16


def _to(a, dtype, dev):
    return torch.tensor(np.ascontiguousarray(a), dtype=dtype, device=dev)


def _f64(t):
    return t.detach().cpu().double().numpy()


def _row_err(a, ref):
    """max over rows of max_i |a - ref| / max_i |ref| (rows = leading axis; exact equality required for a zero row)."""
    if not len(ref):
        return 0.0
    a, ref = np.asarray(a, np.float64).reshape(len(ref), -1), np.asarray(ref, np.float64).reshape(len(ref), -1)
    scale = np.maximum(np.abs(ref).max(axis=1), 1e-300)
    return float((np.abs(a - ref).max(axis=1) / scale).max())


def _ulp_err(a, ref):
    """max over rows of max_i |a - ref| in float32 ulps of the row's largest |ref|."""
    if not len(ref):
        return 0.0
    a, ref = np.asarray(a, np.float64).reshape(len(ref), -1), np.asarray(ref, np.float64).reshape(len(ref), -1)
    ulp = np.spacing(np.abs(ref).max(axis=1).astype(np.float32)).astype(np.float64)
    return float((np.abs(a - ref).max(axis=1) / np.maximum(ulp, 1e-300)).max())


def _check(a, ref, dtype, tol64):
    """float64 outputs within tol64 per row, float32 outputs within 4 ulps of the row maximum."""
    if dtype == torch.float64:
        err = _row_err(a, ref)
        assert err < tol64, "per-row relative error %.3e >= %.1e" % (err, tol64)
    else:
        err = _ulp_err(a, ref)
        assert err <= 4.0, "per-row error %.2f float ulps > 4" % err


def _grid_stride_wrap_batch(d, n):
    """Smallest batch for which both apply kernels' grid-stride loops wrap (their grids are capped at 16 CTAs per SM:
    16 * 256 threads per SM for apply, 16 * 8 warps per SM for apply_T), plus a partial last pass."""
    nsm = torch.cuda.get_device_properties(0).multi_processor_count
    return max(16 * 256 * nsm // d, 16 * 8 * nsm // n) + 5


# ---------------------------------------------------------------------------------------------------------------- apply

@pytest.mark.parametrize("mesh", list(MESHES) + ["synthetic"])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B", [0, 1, 7, 33, 4096, "wrap"])
def test_apply_and_apply_T_against_dense_W(mesh, dtype, B, dev):
    W = _W(mesh)
    d, n = W.shape
    nsm = torch.cuda.get_device_properties(0).multi_processor_count
    if B == "wrap":
        B = _grid_stride_wrap_batch(d, n)
        assert B * d > 16 * 256 * nsm and B * n > 16 * 8 * nsm
    plan = _plan(W, dev)
    rng = np.random.RandomState(B + d)
    u, gy = _to(_dyadic(rng, (B, n)), dtype, dev), _to(rng.normal(size=(B, d)), dtype, dev)
    y, gu = plan.apply(u), plan.apply(gy, transpose=True)
    assert y.shape == (B, d) and gu.shape == (B, n) and y.dtype == gu.dtype == dtype
    y_ref, gu_ref = _f64(u) @ W.T, _f64(gy) @ W
    _check(_f64(y), y_ref, dtype, 1e-14)
    _check(_f64(gu), gu_ref, dtype, 1e-13)
    if B:
        if mesh == "synthetic":            # the empty row and the empty column produce exact zeros
            assert not _f64(y)[:, 5].any() and not _f64(gu)[:, 7].any()
        # adjointness <u W^T, gy> = <u, gy W> of the kernels' own outputs
        lhs, rhs = _f64(y) * _f64(gy), _f64(u) * _f64(gu)
        scale = max(np.abs(lhs).sum(), np.abs(rhs).sum())
        tol = 1e-14 if dtype == torch.float64 else 2.0 ** -22
        assert abs(lhs.sum() - rhs.sum()) <= tol * scale


def test_apply_fp32_beyond_2_pow_31_elements(dev):
    """y [131100, 16383] float32 (8.6 GB, B d > 2^31) on the cfg-3 W: sampled rows, among them the row that crosses
    element 2^31 and the last one, pin the 64-bit indexing of both kernels."""
    W = _W("128x128")
    d, n = W.shape
    B = 131100
    assert B * d > 2 ** 31
    plan = _plan(W, dev)
    gen = torch.Generator(device=dev).manual_seed(7)
    u = torch.round(torch.randn(B, n, device=dev, generator=gen) * 2.0 ** 16) / 2.0 ** 16
    y = plan.apply(u)
    gu = plan.apply(y, transpose=True)
    rows = np.unique(np.concatenate([[0, 1, 2 ** 31 // d - 1, 2 ** 31 // d, 2 ** 31 // d + 1, B - 2, B - 1],
                                     np.random.RandomState(8).randint(0, B, size=40)]))
    idx = torch.tensor(rows, device=dev)
    u_s, y_s, gu_s = _f64(u[idx]), _f64(y[idx]), _f64(gu[idx])
    del y, gu
    torch.cuda.empty_cache()
    _check(y_s, u_s @ W.T, torch.float32, None)
    _check(gu_s, y_s @ W, torch.float32, None)


# ---------------------------------------------------------------------------------------------------------------- loglik

def _loglik_ref(W, u, Y, ls):
    """float64 (L [B], gu [B,n], gls [d], scale [B]) with scale_b = sum_i |2 ls_i + e_bi^2 + log 2 pi|."""
    e = (Y - u @ W.T) * np.exp(-ls)
    terms = 2.0 * ls + e * e + LOG2PI
    return -0.5 * terms.sum(axis=1), (e * np.exp(-ls)) @ W, (e * e - 1.0).sum(axis=0), np.abs(terms).sum(axis=1)


def _loglik_inputs(W, B, seed):
    """Dyadic u, ls in [-8, 3] with both ends present, Y = W u + exp(ls) noise, and one sample 50 sigma off."""
    d, n = W.shape
    rng = np.random.RandomState(seed)
    u = _dyadic(rng, (B, n))
    ls = rng.uniform(-8.0, 3.0, size=d)
    ls[:2] = (-8.0, 3.0)
    Y = u @ W.T + np.exp(ls) * rng.normal(size=(B, d))
    Y[B // 2] += 50.0 * np.exp(ls) * rng.normal(size=d)
    return u, Y, ls


def _check_loglik(W, u, Y, ls, L, gu, gls, dtype):
    """L, gls against the FP64 tolerances for either I/O dtype; gu with _check."""
    L0, gu0, gls0, scale = _loglik_ref(W, _f64(u), _f64(Y), _f64(ls))
    if L is not None:
        err = float((np.abs(_f64(L) - L0) / scale).max())
        assert err < 1e-13, "L: per-sample error %.3e relative to sum_i |terms|" % err
    if gu is not None:
        _check(_f64(gu), gu0, dtype, 1e-13)
    if gls is not None:
        err = _row_err(_f64(gls)[None], gls0[None])
        assert err < 1e-12, "gls: relative error %.3e" % err


@pytest.mark.parametrize("mesh", ["16x16", "32x32", "128x128", "synthetic"])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("B", [1, 7, 8, 9, 31, 32, 33, 65, 128, 320])
def test_loglik_against_float64_reference(mesh, dtype, B, dev):
    """Batches that are not a multiple of the kernel's 8-sample groups, more than one 32-sample chunk (gls summed over
    blockIdx.y), one to four row blocks (d = 255 / 1023), the cfg-3 mesh and the synthetic W."""
    W = _W(mesh)
    plan = _plan(W, dev)
    u, Y, ls = (_to(a, dtype, dev) for a in _loglik_inputs(W, B, B))
    L, gu, gls = plan.loglik(u, Y, ls)
    assert L.dtype == gls.dtype == torch.float64 and gu.dtype == dtype
    _check_loglik(W, u, Y, ls, L, gu, gls, dtype)


def _abi_loglik(plan, u, Y, ls, L, gu, gls, B):
    from gpde_b200 import _lib
    fn = getattr(_lib.load(), "gpde_prolong_loglik_" + _lib.suffix(ls.dtype))
    P = lambda t: _lib.ptr(t, plan.device)
    return fn(plan.handle, P(u), P(Y), P(ls), P(L), P(gu), P(gls), B, _lib.stream_of(plan.device))


@pytest.mark.parametrize("dtype", DTYPES)
def test_loglik_with_null_gu_or_gls(dtype, dev):
    """gu = NULL and gls = NULL each leave the other outputs as the full call computes them."""
    W = _W("32x32")
    d, n = W.shape
    B = 45
    plan = _plan(W, dev)
    u, Y, ls = (_to(a, dtype, dev) for a in _loglik_inputs(W, B, 3))
    L_full, gu_full, gls_full = plan.loglik(u, Y, ls)
    L = torch.full((B,), float("nan"), dtype=torch.float64, device=dev)
    gls = torch.full((d,), float("nan"), dtype=torch.float64, device=dev)
    assert _abi_loglik(plan, u, Y, ls, L, None, gls, B) == 0
    _check_loglik(W, u, Y, ls, L, None, gls, dtype)
    L2 = torch.full((B,), float("nan"), dtype=torch.float64, device=dev)
    gu = torch.full((B, n), float("nan"), dtype=dtype, device=dev)
    assert _abi_loglik(plan, u, Y, ls, L2, gu, None, B) == 0
    _check_loglik(W, u, Y, ls, L2, gu, None, dtype)
    assert torch.equal(gu, gu_full)                            # no atomics in the gu kernel: bitwise
    torch.testing.assert_close(L, L_full, rtol=1e-15, atol=0)
    torch.testing.assert_close(L2, L_full, rtol=1e-15, atol=0)
    torch.testing.assert_close(gls, gls_full, rtol=1e-14, atol=0)


@pytest.mark.parametrize("dtype", DTYPES)
def test_loglik_empty_batch_zeroes_gls(dtype, dev):
    """The header's contract 'L and gls are zeroed by the call' holds for B = 0 too: gls is a sum over the batch."""
    W = _W("32x32")
    d, n = W.shape
    plan = _plan(W, dev)
    u, Y = torch.empty(0, n, dtype=dtype, device=dev), torch.empty(0, d, dtype=dtype, device=dev)
    ls = torch.zeros(d, dtype=dtype, device=dev)
    L, gu = torch.empty(0, dtype=torch.float64, device=dev), torch.empty(0, n, dtype=dtype, device=dev)
    gls = torch.full((d,), float("nan"), dtype=torch.float64, device=dev)
    assert _abi_loglik(plan, u, Y, ls, L, gu, gls, 0) == 0
    assert torch.equal(gls, torch.zeros_like(gls))
    assert _abi_loglik(plan, u, Y, ls, L, gu, None, 0) == 0
    L0, gu0, gls0 = plan.loglik(u, Y, ls)
    assert L0.shape == (0,) and gu0.shape == (0, n) and torch.equal(gls0, torch.zeros_like(gls0))


@pytest.mark.parametrize("dtype", DTYPES)
def test_fused_log_likelihood_of_an_empty_batch_has_zero_gradient(dtype, dev):
    """A rank that gets no samples (sharding.shard_range with B < world) adds exactly zero to the shared gradient of
    logsigmas_y, as the unfused path does -- not whatever memory the caching allocator hands to gls."""
    from gpde_b200.components import ReducedOrderModelOperator
    from oracle import elbo_ref
    op = ReducedOrderModelOperator.FromPhysics(_physics(4, 3), dtype=dtype, device=dev)
    d, n, E = op.dim_out, op.W.shape[1], op.dim_in
    grads = []
    for fused in (True, False):
        # leave NaN-filled blocks of gls's size in the caching allocator
        junk = [torch.full((d,), float("nan"), dtype=torch.float64, device=dev) for _ in range(64)]
        del junk
        eff = torch.zeros(0, E, dtype=dtype, device=dev, requires_grad=True)
        F, Y = torch.zeros(0, n, dtype=dtype, device=dev), torch.zeros(0, d, dtype=dtype, device=dev)
        op.logsigmas_y.grad = None
        if fused:
            L = op.log_likelihood(eff, F, Y)
        else:
            mu, ls = op(eff, F)
            L = elbo_ref.diagonal_gaussian_log_likelihood(Y, mu, 2 * ls)
        L.backward()
        assert L.item() == 0.0
        grads.append(op.logsigmas_y.grad.clone())
    assert torch.equal(grads[0], torch.zeros_like(grads[0]))
    assert torch.equal(grads[0], grads[1])


@pytest.mark.parametrize("n", [200, 799, 800])
def test_loglik_shared_memory_limit(n, dev):
    """The row kernel stages 32 samples x n coarse dofs in shared memory: past the 48 KB default (n > 191) it opts in to
    more, up to 200 KB (n = 799); n = 800 is refused with GPDE_ERR_SIZE before any launch."""
    from gpde_b200._lib import GpdeLibraryError
    W = _synthetic_W(500, n, n)
    plan = _plan(W, dev)
    for dtype in DTYPES:
        u, Y, ls = (_to(a, dtype, dev) for a in _loglik_inputs(W, 37, n))
        if n <= 799:
            L, gu, gls = plan.loglik(u, Y, ls)
            _check_loglik(W, u, Y, ls, L, gu, gls, dtype)
        else:
            with pytest.raises(GpdeLibraryError, match=r"\(-3\)"):
                plan.loglik(u, Y, ls)


# ---------------------------------------------------------------- the fused autograd surface at the 8x8 coarse mesh

@pytest.mark.parametrize("B", [33, 300])
def test_fused_log_likelihood_autograd_on_the_8x8_mesh(B, dev):
    """ReducedOrderModelOperator.log_likelihood (windowed coarse solves with a factor stash + the fused epilogue) against
    CPU float64 autograd through the oracle's operator and Gaussian log-likelihood: value, d/d effprop, d/d F and
    d/d logsigmas_y."""
    from gpde_b200.components import ReducedOrderModelOperator
    from gpde_b200.physics import BoundaryConditionEnsemble
    from oracle import elbo_ref, fem_p1, rom_ref
    ph = _physics(8, 4)
    op = ReducedOrderModelOperator.FromPhysics(ph, dtype=torch.float64, device=dev)
    d, n, E = op.dim_out, op.W.shape[1], op.dim_in
    rng = np.random.RandomState(B)
    c, cells = fem_p1.unit_square_mesh(8, 8)
    M = torch.tensor(fem_p1.rom_element_tensor(c, cells))
    bc = torch.tensor(fem_p1.dirichlet_left_right(c, "ND")[0])
    W = torch.tensor(ph["W"])
    eff0 = rng.normal(0.4, 0.8, size=(B, E))
    F0 = BoundaryConditionEnsemble(ph, B, "ND", rng=rng).FULL_F_WITH_APPLIED_BC("rom") + 0.0
    free = np.setdiff1d(np.arange(n), bc.numpy())
    F0[:, free] = rng.normal(size=(B, free.size)) * 0.1
    ls0 = rng.uniform(-1.5, -0.5, size=d)
    with torch.no_grad():
        mu0 = rom_ref.operator_forward_mean(M, bc, W, torch.tensor(eff0), torch.tensor(F0)).numpy()
    Y0 = mu0 + np.exp(ls0) * rng.normal(size=(B, d))

    with torch.no_grad():
        op.logsigmas_y.copy_(torch.tensor(ls0))
    op.logsigmas_y.grad = None
    eff = torch.tensor(eff0, device=dev, requires_grad=True)
    F = torch.tensor(F0, device=dev, requires_grad=True)
    L = op.log_likelihood(eff, F, torch.tensor(Y0, device=dev))
    (2.5 * L).backward()

    eff_r = torch.tensor(eff0, requires_grad=True)
    F_r = torch.tensor(F0, requires_grad=True)
    ls_r = torch.tensor(ls0, requires_grad=True)
    mu = rom_ref.operator_forward_mean(M, bc, W, eff_r, F_r)
    L_r = elbo_ref.diagonal_gaussian_log_likelihood(torch.tensor(Y0), mu, 2 * ls_r.repeat(B, 1))
    (2.5 * L_r).backward()
    assert abs(L.item() - L_r.item()) <= 1e-10 * abs(L_r.item())
    for got, want in ((eff.grad, eff_r.grad), (F.grad, F_r.grad)):
        err = _row_err(_f64(got), want.numpy())
        assert err < 1e-10, err
    assert _row_err(_f64(op.logsigmas_y.grad)[None], ls_r.grad.numpy()[None]) < 1e-10


# ---------------------------------------------------------------------------------------------------------------- moments

def _moments_ref(W, u, ls):
    """float64 two-pass sample mean / unbiased covariance of u [N,S,n], pushed through W (sparse: W C W^T one data
    point at a time); S = 1 takes the covariance as zero."""
    N, S, n = u.shape
    ubar = u.mean(axis=1)
    uc = u - ubar[:, None, :]
    Ws = scipy.sparse.csr_matrix(W)
    var = np.zeros((N, W.shape[0]))
    if S > 1:
        for k in range(N):
            C = uc[k].T @ uc[k] / (S - 1)
            var[k] = np.asarray(Ws.multiply(Ws @ C).sum(axis=1)).ravel()
    return ubar @ W.T, np.sqrt(var + np.exp(2.0 * ls))


def _check_moments(W, u, ls, y_mean, y_std, dtype, tol_std=1e-12):
    m0, s0 = _moments_ref(W, _f64(u), _f64(ls))
    _check(_f64(y_mean), m0, dtype, 1e-13)
    _check(_f64(y_std), s0, dtype, tol_std)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("N", [1, 3, 128])
@pytest.mark.parametrize("mesh,S", [("32x32", 1), ("32x32", 2), ("32x32", 3), ("32x32", 64), ("32x32", 256),
                                    ("128x128", 1), ("128x128", 2), ("128x128", 64), ("128x128", 234)])
def test_moments_against_float64_reference(mesh, S, N, dtype, dev):
    """n = 25 and n = 81 coarse dofs, S up to the shared-memory limit of the 8x8 mesh; S = 1 gives y_std = exp(ls)."""
    W = _W(mesh)
    d, n = W.shape
    plan = _plan(W, dev)
    rng = np.random.RandomState(N * 1000 + S)
    u = _to(rng.normal(size=(N, 1, n)) + 0.3 * rng.normal(size=(N, S, n)), dtype, dev)
    ls = _to(rng.uniform(-6.0, 1.0, size=d), dtype, dev)
    y_mean, y_std = plan.moments(u, ls)
    assert y_mean.shape == y_std.shape == (N, d) and y_mean.dtype == y_std.dtype == dtype
    _check_moments(W, u, ls, y_mean, y_std, dtype)
    if S == 1:
        assert torch.isfinite(y_std).all()
        _check(_f64(y_std), np.broadcast_to(np.exp(_f64(ls)), (N, d)), dtype, 1e-15)


@pytest.mark.parametrize("mesh,S_max", [("32x32", 998), ("128x128", 234)])
@pytest.mark.parametrize("dtype", DTYPES)
def test_moments_shared_memory_limit(mesh, S_max, dtype, dev):
    """ubar, Cov_u and the S samples must fit in 200 KB of shared memory: S_max passes, S_max + 1 is GPDE_ERR_SIZE."""
    from gpde_b200._lib import GpdeLibraryError
    W = _W(mesh)
    d, n = W.shape
    plan = _plan(W, dev)
    rng = np.random.RandomState(S_max)
    ls = _to(rng.uniform(-4.0, 0.0, size=d), dtype, dev)
    u = _to(rng.normal(size=(2, S_max, n)), dtype, dev)
    y_mean, y_std = plan.moments(u, ls)
    _check_moments(W, u, ls, y_mean, y_std, dtype)
    with pytest.raises(GpdeLibraryError, match=r"\(-3\)"):
        plan.moments(_to(rng.normal(size=(2, S_max + 1, n)), dtype, dev), ls)


def test_moments_of_ill_conditioned_samples(dev):
    """u = 1e5 + 1e-3 noise: the variance is 1e-16 of E[u^2], so a one-pass E[u^2] - E[u]^2 loses it entirely; the
    two-pass kernel keeps y_std within 1e-9 (ls = -30 leaves the sample covariance alone in y_std)."""
    W = _W("32x32")
    d, n = W.shape
    plan = _plan(W, dev)
    rng = np.random.RandomState(4)
    u = _to(1e5 + 1e-3 * rng.normal(size=(3, 64, n)), torch.float64, dev)
    ls = torch.full((d,), -30.0, dtype=torch.float64, device=dev)
    y_mean, y_std = plan.moments(u, ls)
    _check_moments(W, u, ls, y_mean, y_std, torch.float64, tol_std=1e-9)


def test_predictive_moments_on_the_8x8_mesh(dev):
    """ReducedOrderModelOperator.predictive_moments (N = 5, S = 64) against its definition from the coarse solves and a
    dense W: mean and unbiased variance over the samples of W u, plus exp(2 logsigmas_y)."""
    from gpde_b200.components import ReducedOrderModelOperator
    from gpde_b200.physics import BoundaryConditionEnsemble
    ph = _physics(8, 4)
    g = ReducedOrderModelOperator.FromPhysics(ph, dtype=torch.float64, device=dev)
    N, S, E, n = 5, 64, g.dim_in, g.W.shape[1]
    rng = np.random.RandomState(6)
    with torch.no_grad():
        g.logsigmas_y.copy_(_to(rng.normal(size=g.dim_out) * 0.2 - 2.0, torch.float64, dev))
    eff = _to(rng.normal(0.4, 0.5, size=(N, 1, E)) + 0.3 * rng.normal(size=(N, S, E)), torch.float64, dev)
    F = _to(BoundaryConditionEnsemble(ph, N, "ND", rng=rng).FULL_F_WITH_APPLIED_BC("rom"), torch.float64, dev)
    y_mean, y_std = g.predictive_moments(eff, F)
    with torch.no_grad():
        u = g.rom.solve_log(eff.reshape(N * S, E), F[:, None, :].expand(N, S, n).reshape(N * S, n)).reshape(N, S, n)
    mu = np.einsum('sk,nqk->nqs', ph["W"], _f64(u))
    want_mean = mu.mean(axis=1)
    want_std = np.sqrt(mu.var(axis=1, ddof=1) + np.exp(2 * _f64(g.logsigmas_y)))
    assert _row_err(_f64(y_mean), want_mean) < 1e-12
    assert _row_err(_f64(y_std), want_std) < 1e-11


# ------------------------------------------------------------------------------------- the config-5 shapes in FP32

def _cfg5_operator(dev):
    from gpde_b200.components import ReducedOrderModelOperator
    from gpde_b200.workloads import Workload
    from oracle import fem_p1
    w = Workload("cfg1", B=128, seed=3)
    g = ReducedOrderModelOperator.FromPhysics(w.physics, dtype=torch.float32, device=dev)
    c, cells = fem_p1.unit_square_mesh(4, 4)
    M = torch.tensor(fem_p1.rom_element_tensor(c, cells))
    bc = torch.tensor(fem_p1.dirichlet_left_right(c, "ND")[0])
    return w, g, M, bc


def test_cfg5_fused_log_likelihood_fp32(dev):
    """g.log_likelihood at the SVI step's N_s = 128 on the 32x32 mesh in FP32, against float64 autograd through the
    oracle on the same float32 inputs and parameters (W included)."""
    from oracle import elbo_ref, rom_ref
    w, g, M, bc = _cfg5_operator(dev)
    rng = np.random.RandomState(5)
    with torch.no_grad():
        g.logsigmas_y.copy_(_to(rng.uniform(-5.0, -1.0, size=g.dim_out), torch.float32, dev))
    eff = _to(w.logX, torch.float32, dev).requires_grad_(True)
    F = _to(w.F, torch.float32, dev).requires_grad_(True)
    Y = _to(w.y, torch.float32, dev)
    g.logsigmas_y.grad = None
    L = g.log_likelihood(eff, F, Y)
    L.backward()
    eff_r = eff.detach().cpu().double().requires_grad_(True)
    F_r = F.detach().cpu().double().requires_grad_(True)
    ls_r = g.logsigmas_y.detach().cpu().double().requires_grad_(True)
    mu = rom_ref.operator_forward_mean(M, bc, g.W.detach().cpu().double(), eff_r, F_r)
    L_r = elbo_ref.diagonal_gaussian_log_likelihood(Y.cpu().double(), mu, 2 * ls_r.repeat(eff.shape[0], 1))
    L_r.backward()
    e2 = ((Y.cpu().double() - mu.detach()) * torch.exp(-ls_r.detach())) ** 2
    scale = (2 * ls_r.detach() + e2 + LOG2PI).abs().sum().item()
    assert abs(L.item() - L_r.item()) <= 1e-5 * scale
    for got, want in ((eff.grad, eff_r.grad), (F.grad, F_r.grad)):
        err = _row_err(_f64(got), want.numpy())
        assert err < 1e-4, err
    assert _row_err(_f64(g.logsigmas_y.grad)[None], ls_r.grad.numpy()[None]) < 1e-5


def test_cfg5_predictive_moments_fp32(dev):
    """g.predictive_moments at the VO update's N = 128 data points x S = 64 samples in FP32: these numbers go straight
    into the posterior as VO.update(Y_mean, 1 / Y_std^2).  Reference: float64 coarse solves of the same float32 inputs,
    then the moments' definition."""
    from oracle import rom_ref
    w, g, M, bc = _cfg5_operator(dev)
    N, S, E, n = 128, 64, g.dim_in, g.W.shape[1]
    rng = np.random.RandomState(9)
    with torch.no_grad():
        g.logsigmas_y.copy_(_to(rng.uniform(-6.0, -2.0, size=g.dim_out), torch.float32, dev))
    eff = _to(w.logX[:, None, :] + 0.3 * rng.normal(size=(N, S, E)), torch.float32, dev)
    F = _to(w.F, torch.float32, dev)
    y_mean, y_std = g.predictive_moments(eff, F)
    assert y_mean.dtype == y_std.dtype == torch.float32
    u = rom_ref.rom_call(M, bc, torch.exp(eff.cpu().double().reshape(N * S, E)) + 1e-8,
                         F.cpu().double()[:, None, :].expand(N, S, n).reshape(N * S, n)).reshape(N, S, n).numpy()
    m0, s0 = _moments_ref(g.W.cpu().double().numpy(), u, _f64(g.logsigmas_y))
    assert _row_err(_f64(y_mean), m0) < 1e-5
    assert _row_err(_f64(y_std), s0) < 1e-5

"""ReducedOrderModelOperator -- drop-in for bottleneck/components.py:260-323.

forward(effprop, F) = (W @ rom(exp(effprop)+1e-8, F), logsigmas_y.repeat(B,1)), with
  * exp(.)+1e-8, assembly, solve and (in backward) the adjoint in the two ROM kernels (ROM.py here),
  * the prolongation einsum('sk,nk->ns', W, u) as a CSR gather kernel (csrc/prolong.cu): W has <= 3
    non-zeros per row, the reference multiplies by it as a dense [d,n] matrix.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .ROM import ROM


class _ProlongPlan(object):

    def __init__(self, W, device):
        lib = _lib.load()
        device = _lib.require_cuda(device, "ReducedOrderModelOperator")
        W_host = np.ascontiguousarray(W.detach().to("cpu", torch.float64).numpy())
        d, n = W_host.shape
        handle = ctypes.c_void_p()
        rc = lib.gpde_prolong_plan_create(ctypes.byref(handle), d, n, W_host.ctypes.data_as(ctypes.c_void_p),
                                          device.index)
        _lib.check(rc, "gpde_prolong_plan_create")
        self.handle, self.device, self._lib, self.d, self.n = handle, device, lib, d, n

    def __del__(self):
        try:
            if self.handle:
                self._lib.gpde_prolong_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def apply(self, u, transpose=False):
        sfx = _lib.suffix(u.dtype)
        B = u.shape[0]
        out = torch.empty((B, self.n if transpose else self.d), dtype=u.dtype, device=u.device)
        fn = getattr(self._lib, "gpde_prolong_apply_%s%s" % ("T_" if transpose else "", sfx))
        _lib.check(fn(self.handle, _lib.ptr(u, self.device), _lib.ptr(out, self.device), B, _lib.stream_of(self.device)),
                   "gpde_prolong_apply")
        return out


    def loglik(self, u, Y, logsigmas, want_grads=True):
        """(L [B] float64, gu [B,n], gls [d] float64) of the fused epilogue (gpde_prolong_loglik_*): the diagonal-Gaussian
        log-likelihood of Y under N(W u, exp(2 logsigmas)) per sample and its gradients, mu_y = W u never materialised."""
        sfx = _lib.suffix(u.dtype)
        dev, B = self.device, u.shape[0]
        u, Y, ls = u.contiguous(), Y.to(u.dtype).contiguous(), logsigmas.detach().to(u.dtype).contiguous()
        L = torch.empty(B, dtype=torch.float64, device=dev)
        gu = torch.empty_like(u) if want_grads else None
        gls = torch.empty(self.d, dtype=torch.float64, device=dev) if want_grads else None
        fn = getattr(self._lib, "gpde_prolong_loglik_" + sfx)
        _lib.check(fn(self.handle, _lib.ptr(u, dev), _lib.ptr(Y, dev), _lib.ptr(ls, dev), _lib.ptr(L, dev), _lib.ptr(gu, dev),
                      _lib.ptr(gls, dev), B, _lib.stream_of(dev)), "gpde_prolong_loglik")
        return L, gu, gls

    def moments(self, u, logsigmas):
        """(y_mean [N,d], y_std [N,d]) from the coarse solutions u [N,S,n] of S Monte-Carlo samples per data point
        (gpde_prolong_moments_*)."""
        sfx = _lib.suffix(u.dtype)
        dev = self.device
        N, S, n = u.shape
        assert n == self.n
        u, ls = u.contiguous(), logsigmas.detach().to(u.dtype).contiguous()
        y_mean = torch.empty((N, self.d), dtype=u.dtype, device=dev)
        y_std = torch.empty_like(y_mean)
        fn = getattr(self._lib, "gpde_prolong_moments_" + sfx)
        _lib.check(fn(self.handle, _lib.ptr(u, dev), _lib.ptr(ls, dev), _lib.ptr(y_mean, dev), _lib.ptr(y_std, dev), N, S,
                      _lib.stream_of(dev)), "gpde_prolong_moments")
        return y_mean, y_std


class FusedLogLikelihoodFn(torch.autograd.Function):
    """sum_b log N(Y_b | W rom(exp(effprop_b)+1e-8, F_b), exp(2 logsigmas_y)) in three launches (coarse solve, row pass,
    weighted transposed prolongation) and one more in backward (adjoint solve); nothing of size [B,d] is written."""

    @staticmethod
    def forward(ctx, effprop, F, Y, logsigmas, op):
        from .ROM import _launch_forward
        rom, pplan = op.rom, op._prolong_plan()
        plan = rom._get_plan()
        X, Fc = effprop.contiguous(), F.to(effprop.dtype).contiguous()
        need = effprop.requires_grad or F.requires_grad or logsigmas.requires_grad
        u, factor = _launch_forward(plan, X, Fc, True, want_factor=need, info=rom._info_word(X.device))
        L, gu, gls = pplan.loglik(u, Y, logsigmas, want_grads=need)
        ctx.plan = plan
        if need:
            ctx.save_for_backward(X, u, factor if factor is not None else torch.empty(0, device=X.device), gu, gls)
        ctx.ls_dtype = logsigmas.dtype
        return L.sum().to(effprop.dtype)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        from .ROM import _launch_adjoint
        X, u, factor, gu, gls = ctx.saved_tensors
        factor = factor if factor.numel() else None
        gX, gF = _launch_adjoint(ctx.plan, X, u, factor, gu, True, want_gradF=ctx.needs_input_grad[1])
        g = gout.to(X.dtype)
        return (gX * g if ctx.needs_input_grad[0] else None, gF * g if gF is not None else None, None,
                (gls * gout.double()).to(ctx.ls_dtype) if ctx.needs_input_grad[3] else None, None)


class ProlongFn(torch.autograd.Function):
    """y[B,d] = u[B,n] W^T ; backward gbar_u = gbar_y W."""

    @staticmethod
    def forward(ctx, u, plan):
        ctx.plan = plan
        return plan.apply(u.contiguous(), transpose=False)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        return ctx.plan.apply(gy.contiguous(), transpose=True), None


class ReducedOrderModelOperator(torch.nn.Module):

    def __init__(self, rom, W, *, dtype=None, device=None):

        super(ReducedOrderModelOperator, self).__init__()

        self.W = W
        self.rom = rom

        self._dtype = dtype
        self._device = device

        self.logsigmas_y = torch.nn.Parameter(torch.ones(W.shape[0], requires_grad=True))
        self.to(dtype=dtype, device=device)
        self._prolong = None

    @property
    def dtype(self):
        return self._dtype

    @property
    def device(self):
        return self._device

    @property
    def dim_effective_property(self):
        return self.rom.Vc_dim

    @property
    def dim_in(self):
        return self.dim_effective_property

    @property
    def dim_out(self):
        return self.W.shape[0]

    def _prolong_plan(self):
        if self._prolong is None:
            self._prolong = _ProlongPlan(self.W, self.W.device)
        return self._prolong

    def forward(self, effprop, F):

        return self.forward_mean(effprop, F), self.logsigmas_y.repeat(effprop.shape[0], 1)

    def forward_mean(self, effprop, F):

        u = self.rom.solve_log(effprop, F)
        return ProlongFn.apply(u, self._prolong_plan())

    # ------------------------------------------------------------------ fused epilogues (opt-in; SURVEY.md section 8 row f1)
    def log_likelihood(self, effprop, F, Y):
        """DiagonalGaussianLogLikelihood(Y, *self.forward(effprop, F) with logvars = 2 logsigmas_y) (bottleneck/utils.py:231-241,
        the term generative.py:438-439 adds to the ELBO), differentiable in effprop, F and logsigmas_y, WITHOUT the
        intermediate mu_y [B,d]: same value and gradients as the unfused drop-in path up to rounding."""
        out = FusedLogLikelihoodFn.apply(effprop, F, Y, self.logsigmas_y, self)
        if not self.rom.deferred_checks:
            self.rom.check()
        return out

    @torch.no_grad()
    def predictive_moments(self, effprops, F):
        """(Y_mean [N,d], Y_std [N,d]) of the operator output for S samples of the effective property per data point --
        what GenerativeModel.update_virtual_observables computes in a Python loop over data points with
        propagate_samples + torch.mean / torch.std (generative.py:198-207).  effprops [N,S,E], F [N,n].  One batched coarse
        solve and one launch; the output noise is integrated out instead of sampled:
            Y_std^2 = W Cov_s(u) W^T + exp(2 logsigmas_y)  (the expectation of the reference's sample variance).
        S = 1 gives Y_std = exp(logsigmas_y) (no sample covariance; torch.std of one sample would be NaN).  S is limited by
        shared memory: S <= 998 on the 4x4 coarse mesh, S <= 234 on the 8x8 one (GpdeLibraryError beyond)."""
        N, S, E = effprops.shape
        Fx = F.unsqueeze(1).expand(N, S, F.shape[-1]).reshape(N * S, -1)
        u = self.rom.solve_log(effprops.reshape(N * S, E), Fx)
        return self._prolong_plan().moments(u.reshape(N, S, -1), self.logsigmas_y)

    def propagate_samples(self, effprops, F):

        means, logsigmas = self.forward(effprops, F)

        if means.shape != logsigmas.shape:
            raise RuntimeError('Implementation assumes that full logsigmas matrix is given; check for broadcasting')

        return means + torch.exp(logsigmas) * torch.randn_like(logsigmas)

    @classmethod
    def FromPhysics(cls, physics, *, dtype=None, device=None):

        W = torch.tensor(physics['W'].T, dtype=dtype, device=device).t()

        if W.shape[0] < W.shape[1]:
            raise ValueError

        rom = ROM.FromPhysics(physics['rom'], dtype=dtype, device=device)
        return cls(rom, W, dtype=dtype, device=device)

"""Virtual observables for the B200 physics layer (API surface of bottleneck/VirtualObservables.py).

Design (not the reference's): the reference keeps one Python object per data point, each holding a
dense Gamma = V^T K assembled on the CPU from a FEniCS/scipy CSR matrix, and loops over them
(VirtualObservables.py:61-69, 642-669, 891-898, 971-998).  Here

  * the fine operator is never assembled: r = V^T (K_fom(a) u~ - f) and q = K_ff(a) (V s) are launches
    of the matrix-free kernels in csrc/vo.cu (``VoPlan.residual`` / ``VoPlan.residual_T``);
  * Gamma and alpha, where the reference API exposes them, are produced on the device by those same
    kernels: Gamma^T = K_ff V is ``residual_T`` applied to the identity, alpha = -r(y = 0);
  * an ensemble conditions all its data points in one batched pass (``condition_gaussian``) and
    evaluates all residuals in one launch; the per-data-point classes are thin views kept for
    callers that index into the ensemble (generative.py:198-207, training.py:320-339).

The names the reference's callers use are kept: QuerryPoint(.x/.bc/.K/.f/.construct_querry_weak_galerkin),
QuerryPointEnsemble, the samplers, LinearQuerry(.Gamma/.GammaTransposed/.alpha/.m/.resample),
QuerryEnsemble.FromQuerryPointEnsemble, VirtualObservable(.update/.mean/.vars/.vo_variances),
VirtualObservablesEnsemble(.update/.mean/.vars/.logsigma/.resample/.N/.m/.dim_out) and the temperature
schedules.  Flux test functions (bottleneck/flux.py) need UFL facet integrals and stay out of scope.
"""
import ctypes
import os

import numpy as np
import torch

from . import _lib
from . import fem

_F64 = torch.float64


def _as_f64(value, device):
    return torch.as_tensor(value, dtype=_F64, device=device)


# ======================================================================================= device plan
class VoPlan(object):
    """One gpde_vo_plan: fine-mesh element data and the Dirichlet map, resident on a device."""

    def __init__(self, physics, device, cell_to_input=None, n_inputs=None, load=None, experiment=None):
        self._lib = _lib.load()
        self.device = _lib.require_cuda(device, "virtual observables")
        self._ctor = (physics, cell_to_input, n_inputs, load)
        self.cell_to_input = None if cell_to_input is None else np.asarray(cell_to_input)
        mesh = physics.mesh
        if cell_to_input is None:
            cell_to_input, n_inputs = np.arange(mesh.num_cells), mesh.num_cells
        host = dict(
            cells=np.ascontiguousarray(mesh.cells, dtype=np.int32),
            Ke=np.ascontiguousarray(mesh.element_stiffness(), dtype=np.float64),
            c2i=np.ascontiguousarray(cell_to_input, dtype=np.int32),
            free=np.ascontiguousarray(physics.free_dofs, dtype=np.int64),
            bc=np.ascontiguousarray(physics.constrained_dofs, dtype=np.int64),
        )
        if load is not None:
            host["load"] = np.ascontiguousarray(load, dtype=np.float64)
        p = {k: v.ctypes.data_as(ctypes.c_void_p) for k, v in host.items()}
        self.handle = ctypes.c_void_p()
        # the library reads its experiment switches (GPDE_* environment variables, A/B runs of the kernel families) ONCE,
        # here; ``experiment`` sets them for this plan only
        saved = {k: os.environ.get(k) for k in (experiment or {})}
        os.environ.update({k: str(v) for k, v in (experiment or {}).items()})
        try:
            rc = self._lib.gpde_vo_plan_create(ctypes.byref(self.handle), mesh.num_nodes, mesh.num_cells, p["cells"],
                                               p["Ke"], p["c2i"], int(n_inputs), p["free"], host["free"].size, p["bc"],
                                               host["bc"].size, p.get("load"), self.device.index)
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        _lib.check(rc, "gpde_vo_plan_create")
        info = (ctypes.c_int64 * 8)()
        _lib.check(self._lib.gpde_vo_plan_info(self.handle, info), "gpde_vo_plan_info")
        self.n_nodes, self.n_cells, self.n_inputs, self.d, self.n_bc, self.slots_per_row = (int(v) for v in info[:6])
        self.fused_smem_bytes = int(info[7])   # 0: this mesh only runs on the unfused version-1 kernels
        self._scratch = None

    def __del__(self):
        handle, self.handle = getattr(self, "handle", None), None
        if handle:
            try:
                self._lib.gpde_vo_plan_destroy(handle)
            except Exception:
                pass

    def variant(self, **experiment):
        """A second plan on the same mesh data with experiment switches (tests and A/B timing runs)."""
        physics, c2i, n_in, load = self._ctor
        return VoPlan(physics, self.device, c2i, n_in, load, experiment=experiment)

    @classmethod
    def cached(cls, physics, device, pixel_input=False):
        """Plans are immutable; one per (physics, device, input layout) is kept on the physics object."""
        device = _lib.require_cuda(device, "virtual observables")
        store = physics.__dict__.setdefault("_gpde_vo_plans", {})
        key = (device.index, bool(pixel_input))
        if key not in store:
            if pixel_input:
                store[key] = cls(physics, device, physics.mesh.pixel_of_cell(), physics.mesh.nx * physics.mesh.ny)
            else:
                store[key] = cls(physics, device)
        return store[key]

    def kernel_path(self, m, dtype=torch.float64):
        """3 = grid rho kernel + tensor-core contraction (m > 32), 2 = structured-grid kernel, 1 = generic fused
        kernel, 0 = version-1 kernels (include/gpde_b200.h)."""
        return int(self._lib.gpde_vo_plan_kernel_path(self.handle, int(m), 8 if dtype == torch.float64 else 4))

    def launches_per_residual(self, m, dtype=torch.float64):
        """Kernels launched by one residual() call (for bench.py's gpu_launches count)."""
        path = self.kernel_path(m, dtype)
        return {3: 3, 2: 2, 1: 1}.get(path, 3 if m > 0 else 1)

    def _workspace(self, B, m):
        need = max(16, int(self._lib.gpde_vo_workspace_bytes(self.handle, B, m)))
        if self._scratch is None or self._scratch.numel() < need:
            self._scratch = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._scratch

    def pack_weights(self, V, B, *, ignore_load=False, out=None):
        """Packs V [d,m] once for many residual() calls with the same weighting functions (V = W of the
        coarse-grained-residual sampler only changes at resample()).  Returns a PackedWeights to pass as ``V``,
        or V itself when this plan / m has no packed layout.  B = the largest batch it will be used with;
        ``out`` = an earlier PackedWeights whose buffer is reused."""
        if V.dim() != 2:
            raise ValueError("pack_weights packs one weighting matrix [d,m] shared by the batch, got V of shape %r"
                             % (tuple(V.shape),))
        dt = V.dtype if V.dtype in (torch.float32, torch.float64) else torch.float64
        Vc = V.to(dt).contiguous()
        sfx = _lib.suffix(dt)
        m = int(Vc.shape[1])
        need = max(8, int(self._lib.gpde_vo_workspace_bytes(self.handle, int(B), m)))
        if out is not None and out.buf.numel() >= need:
            buf = out.buf
        else:
            buf = torch.empty(need, dtype=torch.uint8, device=self.device)
        rc = getattr(self._lib, "gpde_vo_pack_weights_" + sfx)(self.handle, _lib.ptr(Vc, self.device), m, 1 if ignore_load else 0,
                                                               _lib.ptr(buf, self.device), _lib.stream_of(self.device))
        if rc == 1:
            return Vc
        _lib.check(rc, "gpde_vo_pack_weights_" + sfx)
        return PackedWeights(Vc, buf, int(B), bool(ignore_load))

    def residual(self, a, y, g, V, *, a_is_log=True, want_rho=False, ignore_load=False, sm_reserve=0):
        """r[B,m] = V^T (K(a_b) u~_b - f)_free with u~ = (y on free dofs, g on Dirichlet dofs).

        a [B,n_inputs] or [n_inputs] (shared); y [B,d] or None (zeros); g [B,n_bc], [n_bc] or None;
        V [d,m] shared by the batch, [B,d,m] one matrix per sample (r_b = V_b^T rho_b), or None (then only rho[B,d], the
        fine residual itself, is produced).
        Returns r, or (r, rho) when want_rho / V is None.
        ``sm_reserve``: SMs to leave to kernels the caller runs beside this call on other streams (the structured-grid
        kernel sizes its last wave of CTAs for the remaining SMs; a [B,d,m] V has no such kernel and ignores it)."""
        dt = a.dtype
        sfx = _lib.suffix(dt)
        per_sample = V is not None and not isinstance(V, PackedWeights) and V.dim() == 3
        sizes = [t.shape[0] for t in (y, a, g) if t is not None and t.dim() == 2]
        B = sizes[0] if sizes else (int(V.shape[0]) if per_sample else 1)
        if any(n != B for n in sizes):   # e.g. a shared 1-D field with y = None and a batched g: every batched argument counts
            raise ValueError("inconsistent batch sizes %r among a, y, g" % (sizes,))
        a = a.contiguous()
        packed = None
        if isinstance(V, PackedWeights):
            # usable as packed only for the kind of call it was packed for; otherwise the plain matrix is used
            if (dt == V.V.dtype and y is not None and not want_rho and B <= V.B and V.ignore_load == bool(ignore_load)
                    and a.data_ptr() % 16 == 0):
                packed = V
            V = V.V
        y = None if y is None else y.to(dt).contiguous()
        g = None if g is None else g.to(dt).contiguous()
        Vc, v_stride, m = (None, 0, 0) if V is None else self._weights_arg(V, dt, B)
        r = a.new_empty((B, m)) if m else None
        rho = a.new_empty((B, self.d)) if (want_rho or not m) else None
        fn = getattr(self._lib, "gpde_vo_residual_" + sfx)
        ws = packed.buf if packed is not None else (self._workspace(B, m) if m else None)
        dev = self.device
        rc = fn(self.handle, _lib.ptr(a, dev), self.n_inputs if a.dim() == 2 else 0, int(bool(a_is_log)), _lib.ptr(y, dev),
                _lib.ptr(g, dev), (self.n_bc if g.dim() == 2 else 0) if g is not None else 0, _lib.ptr(Vc, dev), v_stride, m,
                _lib.ptr(r, dev), _lib.ptr(rho, dev), _lib.ptr(ws, dev) if m else None,
                (1 if ignore_load else 0) | (2 if packed is not None else 0) | (max(0, min(255, int(sm_reserve))) << 8), B,
                _lib.stream_of(dev))
        _lib.check(rc, "gpde_vo_residual_" + sfx)
        return (r, rho) if rho is not None else r

    def _weights_arg(self, V, dt, B):
        """(contiguous V in dt, v_stride, m): V [d,m] shared by the batch (v_stride = 0) or [B,d,m] one matrix per sample
        (v_stride = d*m); ValueError unless a [B,d,m] V matches the batch size B and the plan."""
        if V.dim() == 2:
            return V.to(dt).contiguous(), 0, int(V.shape[1])
        if V.dim() != 3 or V.shape[0] != B or V.shape[1] != self.d or V.shape[2] < 1:
            raise ValueError("per-sample weighting matrices must be [B=%d, d=%d, m>=1], got %r" % (B, self.d, tuple(V.shape)))
        return V.to(dt).contiguous(), int(V.shape[1] * V.shape[2]), int(V.shape[2])

    def residual_T(self, a, V, s, *, a_is_log=True):
        """q[B,d] = K_ff(a_b) (V s_b)  (= Gamma_b^T s_b); V [d,m] shared by the batch or [B,d,m] one matrix per sample
        (q_b = K_ff(a_b) (V_b s_b))."""
        dt = a.dtype
        sfx = _lib.suffix(dt)
        dev = self.device
        a, s = a.contiguous(), s.to(dt).contiguous()
        B, m = int(s.shape[0]), int(s.shape[1])
        Vc, v_stride, mv = self._weights_arg(V, dt, B)
        if v_stride and ((a.dim() == 2 and a.shape[0] != B) or mv != m):
            raise ValueError("inconsistent shapes: a %r, V %r, s %r" % (tuple(a.shape), tuple(V.shape), tuple(s.shape)))
        q = a.new_empty((B, self.d))
        fn = getattr(self._lib, "gpde_vo_residual_T_" + sfx)
        rc = fn(self.handle, _lib.ptr(a, dev), self.n_inputs if a.dim() == 2 else 0, int(bool(a_is_log)), _lib.ptr(Vc, dev),
                v_stride, m, _lib.ptr(s, dev), _lib.ptr(q, dev), _lib.ptr(self._workspace(B, m), dev), B, _lib.stream_of(dev))
        _lib.check(rc, "gpde_vo_residual_T_" + sfx)
        return q

    def residual_grad(self, a, y, g, V, gbar_r, *, a_is_log=True, want_grad_a=True, want_grad_g=False):
        """(grad_a, grad_g): the gradient of L with dL/dr = gbar_r [B,m] through r = residual(a, y, g, V) with respect to
        the conductivity input a and the Dirichlet values g (gpde_vo_residual_grad_*; r is linear in both, no solve):
            grad_a[b,p] = sum_{cells c of input p} w~_b[c]^T K_c u~_b[c],   grad_g[b] = K_cf(a_b) w~_b,
        w~_b = V gbar_r_b on the free dofs (0 on the Dirichlet dofs); V [d,m] shared by the batch or [B,d,m] one matrix per
        sample (w~_b = V_b gbar_r_b).  With ``a_is_log`` a = exp(x) and grad_a is the gradient in x.  A gradient that is not
        wanted is None.  For a shared 1-D ``a`` or ``g`` the per-sample gradients are summed over the batch.  The load
        vector does not enter."""
        dt = a.dtype
        sfx = _lib.suffix(dt)
        dev = self.device
        gbar_r = gbar_r.to(dt).contiguous()
        B, m = int(gbar_r.shape[0]), int(gbar_r.shape[1])
        sizes = [t.shape[0] for t in (y, a, g) if t is not None and t.dim() == 2]
        if any(n != B for n in sizes):   # the kernels index every batched argument by the B of gbar_r
            raise ValueError("inconsistent batch sizes %r among a, y, g and gbar_r (%d)" % (sizes, B))
        a = a.contiguous()
        y = None if y is None else y.to(dt).contiguous()
        g = None if g is None else g.to(dt).contiguous()
        Vc, v_stride, mv = self._weights_arg(V, dt, B)
        if v_stride and mv != m:
            raise ValueError("gbar_r has %d columns, V_b %d" % (m, mv))
        grad_a = a.new_empty((B, self.n_inputs)) if want_grad_a else None
        grad_g = a.new_empty((B, self.n_bc)) if want_grad_g else None
        fn = getattr(self._lib, "gpde_vo_residual_grad_" + sfx)
        rc = fn(self.handle, _lib.ptr(a, dev), self.n_inputs if a.dim() == 2 else 0, int(bool(a_is_log)), _lib.ptr(y, dev),
                _lib.ptr(g, dev), (self.n_bc if g.dim() == 2 else 0) if g is not None else 0, _lib.ptr(Vc, dev), v_stride, m,
                _lib.ptr(gbar_r, dev), _lib.ptr(grad_a, dev), _lib.ptr(grad_g, dev), _lib.ptr(self._workspace(B, m), dev),
                B, _lib.stream_of(dev))
        _lib.check(rc, "gpde_vo_residual_grad_" + sfx)
        if grad_a is not None and a.dim() == 1:
            grad_a = grad_a.sum(0)
        if grad_g is not None and g is not None and g.dim() == 1:
            grad_g = grad_g.sum(0)
        return grad_a, grad_g

    def posterior(self, a, V, rho, noise_var, g, prec, info=None):
        """Gaussian conditioning of N data points in ONE launch, matrix-free (gpde_vo_posterior_f64):
        (mean [N,d], vars [N,d]) of N(g, diag(1/prec)) given Gamma y = alpha + eps, eps ~ N(0, diag(noise_var)), with
        Gamma^T = K_ff(a_n) V_n never stored.  a: conductivities [N,n_inputs] (or one shared field), rho [N,d] the fine
        residual of the prior mean (``residual(a, g, g_bc, None)``), V [d,m] or [N,d,m]."""
        dev = self.device
        N = int(g.shape[0])
        a = a.to(torch.float64).contiguous()
        V, v_stride, m = self._weights_arg(V, torch.float64, N)
        rho, g, prec = (t.to(torch.float64).contiguous() for t in (rho, g, prec))
        noise_var = noise_var.to(torch.float64).contiguous()
        mean, vars_ = torch.empty_like(g), torch.empty_like(g)
        rc = self._lib.gpde_vo_posterior_f64(self.handle, _lib.ptr(a, dev), self.n_inputs if a.dim() == 2 else 0,
                                             _lib.ptr(V, dev), v_stride, m, _lib.ptr(rho, dev), _lib.ptr(noise_var, dev),
                                             _lib.ptr(g, dev), _lib.ptr(prec, dev), _lib.ptr(mean, dev), _lib.ptr(vars_, dev),
                                             _lib.ptr(info, dev), N, _lib.stream_of(dev))
        _lib.check(rc, "gpde_vo_posterior_f64")
        return mean, vars_

    def posterior_blocked(self, a, V, rho, noise_var, g, prec, info=None):
        """``posterior`` for 1 <= m <= 256 (gpde_vo_posterior_blocked_f64): Lambda_n and L_n^-1 live in a workspace this call
        allocates (about 1 MB per data point at m = 256) instead of shared memory; three launches for all data points."""
        dev = self.device
        N = int(g.shape[0])
        a = a.to(torch.float64).contiguous()
        V, v_stride, m = self._weights_arg(V, torch.float64, N)
        rho, g, prec = (t.to(torch.float64).contiguous() for t in (rho, g, prec))
        noise_var = noise_var.to(torch.float64).contiguous()
        mean, vars_ = torch.empty_like(g), torch.empty_like(g)
        need = int(self._lib.gpde_vo_posterior_blocked_workspace_bytes(self.handle, N, m))
        ws = torch.empty(max(need, 16), dtype=torch.uint8, device=dev)
        rc = self._lib.gpde_vo_posterior_blocked_f64(self.handle, _lib.ptr(a, dev), self.n_inputs if a.dim() == 2 else 0,
                                                     _lib.ptr(V, dev), v_stride, m, _lib.ptr(rho, dev),
                                                     _lib.ptr(noise_var, dev), _lib.ptr(g, dev), _lib.ptr(prec, dev),
                                                     _lib.ptr(mean, dev), _lib.ptr(vars_, dev), _lib.ptr(info, dev),
                                                     _lib.ptr(ws, dev), need, N, _lib.stream_of(dev))
        _lib.check(rc, "gpde_vo_posterior_blocked_f64")
        return mean, vars_

    def posterior_blocked_workspace_bytes(self, N, m):
        return int(self._lib.gpde_vo_posterior_blocked_workspace_bytes(self.handle, int(N), int(m)))

    def moments(self, a, V, rho, v):
        """(r [N,m], s2 [N,m]) = (V_n^T rho_n, sum_i Gamma_n[:,i]^2 v[n,i]) for all data points in one launch
        (gpde_vo_moments_f64, m <= 256): the two terms of the precision hyper-update (VirtualObservables.py:985-990)."""
        dev = self.device
        N = int(rho.shape[0])
        a = a.to(torch.float64).contiguous()
        V, v_stride, m = self._weights_arg(V, torch.float64, N)
        rho, v = rho.to(torch.float64).contiguous(), v.to(torch.float64).contiguous()
        out_r, out_s2 = rho.new_empty((N, m)), rho.new_empty((N, m))
        rc = self._lib.gpde_vo_moments_f64(self.handle, _lib.ptr(a, dev), self.n_inputs if a.dim() == 2 else 0,
                                           _lib.ptr(V, dev), v_stride, m, _lib.ptr(rho, dev), _lib.ptr(v, dev),
                                           _lib.ptr(out_r, dev), _lib.ptr(out_s2, dev), N, _lib.stream_of(dev))
        _lib.check(rc, "gpde_vo_moments_f64")
        return out_r, out_s2

    def energy_step(self, a, V, rho, g, prec, inv_T, mean, info=None):
        """One subspace-Newton step of the energy-type virtual observables for N data points in ONE launch, matrix-free
        (gpde_vo_energy_step_f64), in place on ``mean`` [N,d] (contiguous float64 on this device):
            mean_n <- mean_n - V_n M_n^-1 V_n^T (prec_n (mean_n - g_n) + inv_T[n] rho_n),
            M_n = V_n^T diag(prec_n) V_n + inv_T[n] V_n^T K_ff(a_n) V_n.
        a: conductivities [N,n_inputs] (or one shared field), V [d,m] or [N,d,m] (m <= 64), rho [N,d] = K_ff(a_n) mean_n
        - f_eff (``residual(a, mean, g_bc, None)`` minus the load), g, prec [N,d], inv_T [N].  A data point whose M_n has a
        non-positive pivot keeps its mean and sets GPDE_INFO_NOT_SPD in ``info``.  Returns ``mean``."""
        dev = self.device
        N, a, V, v_stride, m, rho, g, prec, inv_T = self._energy_operands("energy_step", a, V, rho, g, prec, inv_T, mean)
        rc = self._lib.gpde_vo_energy_step_f64(self.handle, _lib.ptr(a, dev), self.n_inputs if a.dim() == 2 else 0,
                                               _lib.ptr(V, dev), v_stride, m, _lib.ptr(rho, dev), _lib.ptr(g, dev),
                                               _lib.ptr(prec, dev), _lib.ptr(inv_T, dev), _lib.ptr(mean, dev),
                                               _lib.ptr(info, dev), N, _lib.stream_of(dev))
        _lib.check(rc, "gpde_vo_energy_step_f64")
        return mean

    def energy_step_blocked(self, a, V, rho, g, prec, inv_T, mean, info=None):
        """``energy_step`` for 1 <= m <= 256 (gpde_vo_energy_step_blocked_f64): M_n lives in a workspace this call
        allocates (the blocked posterior's, about 1 MB per data point at m = 256) instead of shared memory; three launches
        for all data points.  Same arguments, checks and in-place update of ``mean``; returns ``mean``."""
        dev = self.device
        N, a, V, v_stride, m, rho, g, prec, inv_T = self._energy_operands("energy_step_blocked", a, V, rho, g, prec, inv_T,
                                                                          mean)
        need = int(self._lib.gpde_vo_posterior_blocked_workspace_bytes(self.handle, N, m))
        ws = torch.empty(max(need, 16), dtype=torch.uint8, device=dev)
        rc = self._lib.gpde_vo_energy_step_blocked_f64(self.handle, _lib.ptr(a, dev), self.n_inputs if a.dim() == 2 else 0,
                                                       _lib.ptr(V, dev), v_stride, m, _lib.ptr(rho, dev), _lib.ptr(g, dev),
                                                       _lib.ptr(prec, dev), _lib.ptr(inv_T, dev), _lib.ptr(mean, dev),
                                                       _lib.ptr(info, dev), _lib.ptr(ws, dev), need, N,
                                                       _lib.stream_of(dev))
        _lib.check(rc, "gpde_vo_energy_step_blocked_f64")
        return mean

    def _energy_operands(self, name, a, V, rho, g, prec, inv_T, mean):
        """(N, a, V, v_stride, m, rho, g, prec, inv_T) of an energy step, as contiguous float64, with the shape checks."""
        if not (mean.dtype == torch.float64 and mean.dim() == 2 and mean.is_contiguous()):
            raise ValueError("%s updates mean in place: it must be a contiguous float64 [N,d] tensor" % name)
        N = int(mean.shape[0])
        a = a.to(torch.float64).contiguous()
        V, v_stride, m = self._weights_arg(V, torch.float64, N)
        rho, g, prec = (t.to(torch.float64).contiguous() for t in (rho, g, prec))
        inv_T = torch.as_tensor(inv_T, dtype=torch.float64, device=self.device).contiguous()
        if any(t.shape != mean.shape for t in (rho, g, prec)) or mean.shape[1] != self.d or inv_T.shape != (N,) or \
                (a.dim() == 2 and a.shape[0] != N):
            raise ValueError("%s: inconsistent shapes" % name)
        return N, a, V, v_stride, m, rho, g, prec, inv_T


class PackedWeights(object):
    """V [d,m] together with its fragment-packed copy (VoPlan.pack_weights); accepted wherever residual() takes V."""

    def __init__(self, V, buf, B, ignore_load):
        self.V, self.buf, self.B, self.ignore_load = V, buf, B, ignore_load

    @property
    def shape(self):
        return self.V.shape


class VoResidualFn(torch.autograd.Function):
    """r = V^T (K(a) u~ - f), differentiable in y: dL/dy = K_ff(a) V gbar_r (one residual_T call), in the
    conductivity input a and in the Dirichlet values g (VoPlan.residual_grad).  V [d,m] shared by the batch or [B,d,m]
    one matrix per sample (passed through to every call as it is).  V gets no gradient (None)."""

    @staticmethod
    def forward(ctx, y, a, g, V, plan, a_is_log):
        ctx.plan, ctx.a_is_log = plan, a_is_log
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            ctx.save_for_backward(a, V, y, g)
        else:
            ctx.save_for_backward(a, V)
        return plan.residual(a, y, g, V, a_is_log=a_is_log)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gbar_r):
        a, V = ctx.saved_tensors[:2]
        grad_y = grad_a = grad_g = None
        if ctx.needs_input_grad[0]:
            grad_y = ctx.plan.residual_T(a, V, gbar_r.contiguous(), a_is_log=ctx.a_is_log)
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            y, g = ctx.saved_tensors[2:]
            grad_a, grad_g = ctx.plan.residual_grad(a, y, g, V, gbar_r, a_is_log=ctx.a_is_log,
                                                    want_grad_a=ctx.needs_input_grad[1], want_grad_g=ctx.needs_input_grad[2])
            if grad_g is not None:
                grad_g = grad_g.to(g.dtype)
        return grad_y, grad_a, grad_g, None, None, None


def condition_gaussian(Gamma, alpha, noise_var, g, prec):
    """Posterior of y ~ N(g, diag(1/prec)) given Gamma y = alpha + eps, eps ~ N(0, diag(noise_var)).

    Batched over the leading axis: Gamma [N,m,d], alpha [N,m], noise_var [m], g/prec [N,d].
    Same algebra as VirtualObservable.update (VirtualObservables.py:656-669):
        Lambda = Gamma C Gamma^T + Sigma,  mean = g - C Gamma^T Lambda^-1 (Gamma g - alpha),
        vars = diag(C) - diag(C Gamma^T Lambda^-1 Gamma C)."""
    C = 1.0 / prec
    GC = Gamma * C.unsqueeze(-2)                                   # [N,m,d]
    Lam = GC @ Gamma.transpose(-1, -2) + torch.diag(noise_var)
    chol = torch.linalg.cholesky(Lam)
    resid = (Gamma @ g.unsqueeze(-1)).squeeze(-1) - alpha          # [N,m]
    sol = torch.cholesky_solve(resid.unsqueeze(-1), chol)          # Lambda^-1 resid
    mean = g - (GC.transpose(-1, -2) @ sol).squeeze(-1)
    Z = torch.cholesky_solve(GC, chol)                             # Lambda^-1 Gamma C
    return mean, C - (GC * Z).sum(dim=-2)


# ======================================================================================= query points
class QuerryPoint(object):
    """One data point of the virtual-observable set: fine log-conductivity ``x`` (one value per DG0
    cell) and its boundary condition ``bc``   (VirtualObservables.py:8-69)."""

    def __init__(self, physics, x, bc, device=None):
        assert isinstance(x, np.ndarray) and x.ndim == 1
        assert not isinstance(physics, dict)
        assert physics.dim_in == x.size
        self._physics, self._x, self._bc, self._device = physics, x, bc, device
        self._host_system = None

    physics = property(lambda self: self._physics)
    bc = property(lambda self: self._bc)
    x = property(lambda self: self._x, doc="log-conductivity (the reference's naming)")
    dim_in = property(lambda self: self._x.size)
    dim_out = property(lambda self: self._physics.dim_out)

    def _assemble_system(self):
        # host scipy CSR, API parity only (VirtualObservables.py:57-59); the device path never forms K
        if self._host_system is None:
            self._host_system = self._physics.assemble_system(np.exp(self._x), bc=self._bc, only_free_dofs=True)
        return self._host_system

    K = property(lambda self: self._assemble_system()[0])
    f = property(lambda self: self._assemble_system()[1])

    def dirichlet_values(self):
        return self._bc.constrained_dofs_values(self._physics.identifier)

    def weak_galerkin_on_device(self, V, device=None):
        """(Gamma [m,d], alpha [m]) as float64 device tensors via the matrix-free kernels."""
        device = device if device is not None else self._device
        if device is None and torch.cuda.is_available():
            device = torch.device("cuda", torch.cuda.current_device())
        device = _lib.require_cuda(device if device is not None else "cpu", "QuerryPoint")
        plan = VoPlan.cached(self._physics, device)
        Vd = _as_f64(V, device)
        assert Vd.shape[0] == self.dim_out
        a = _as_f64(self._x, device)
        Gamma = plan.residual_T(a, Vd, torch.eye(Vd.shape[1], dtype=_F64, device=device))
        alpha = -plan.residual(a, None, _as_f64(self.dirichlet_values(), device), Vd)
        load = self._bc.assemble_vanilla_force_vector(self._physics.identifier)
        if np.any(load != 0):   # the cached plan carries no load vector: add V^T f_free
            alpha = alpha + Vd.t() @ _as_f64(load[self._physics.free_dofs], device)
        return Gamma, alpha.reshape(-1)

    def construct_querry_weak_galerkin(self, V):
        """numpy (Gamma, alpha) like VirtualObservables.py:61-69."""
        Gamma, alpha = self.weak_galerkin_on_device(V)
        return Gamma.cpu().numpy(), alpha.cpu().numpy()


class QuerryPointEnsemble(object):
    """VirtualObservables.py:72-116."""

    def __init__(self, QPs):
        self._QPs = list(QPs)

    def __iter__(self):
        return iter(self._QPs)

    def __getitem__(self, item):
        return self._QPs[item]

    def __len__(self):
        return len(self._QPs)

    N = property(lambda self: len(self._QPs))
    dim_out = property(lambda self: self._QPs[0].dim_out)

    def X(self, dtype, device):
        return torch.tensor(np.stack([qp.x for qp in self._QPs]), dtype=dtype, device=device)

    def dirichlet_values(self, dtype, device):
        return torch.tensor(np.stack([qp.dirichlet_values() for qp in self._QPs]), dtype=dtype, device=device)

    @classmethod
    def FromArrays(cls, X_DG, BCE, physics, device=None):
        X_DG = X_DG.detach().cpu().numpy() if isinstance(X_DG, torch.Tensor) else np.asarray(X_DG)
        assert X_DG.dtype == np.float64
        return cls(QuerryPoint(physics, X_DG[n].ravel(), BCE[n], device=device) for n in range(X_DG.shape[0]))

    @classmethod
    def FromDataSet(cls, dataset, physics):
        X_DG = dataset.get('X_DG')
        assert X_DG.dtype == torch.double
        return cls.FromArrays(X_DG, dataset.get('BCE'), physics)


# ======================================================================================= samplers
class BaseSampler(object):
    """Produces the weighting matrix V [d,m] of one data point and its (Gamma, alpha).
    precision_mask: -1 = infinite precision, +1 = learnable (VirtualObservables.py:120-168)."""

    is_constant = False
    provides_V = True     # False: the sampler only has (Gamma, alpha) (flux constraints); the ensemble then conditions densely

    def __init__(self, qp):
        self._qp = qp

    qp = property(lambda self: self._qp)
    dim = property(lambda self: self.qp.dim_out)
    fixed_precision = property(lambda self: bool(np.all(self.precision_mask < 0)))
    precision_mask = property(lambda self: -np.ones(self.m))

    def sample_V(self):
        return self._sample()

    def sample_V_batch(self, count):
        """[count, d, m]: ``count`` successive sample_V() draws, stacked in draw order (a numpy array when every draw is
        one, else a float64 tensor on the draws' device)."""
        Vs = [self.sample_V() for _ in range(count)]
        if all(isinstance(v, np.ndarray) for v in Vs):
            return np.stack(Vs)
        device = next(v.device for v in Vs if isinstance(v, torch.Tensor))
        return torch.stack([_as_f64(v, device) for v in Vs])

    def sample(self):
        return self.qp.weak_galerkin_on_device(self._sample())

    def __call__(self):
        return self.sample()


class ConstLengthScaleGenerator(object):
    def __init__(self, l):
        self._l = l

    def __call__(self):
        return self._l


class RadialBasisFunctionSampler(BaseSampler):
    """exp(-|x-r0|^2/l^2) with r0 ~ U[0,1]^2 at the fine free nodes (VirtualObservables.py:172-228,
    fawkes/Expressions.py:26-31): nodal interpolation of a P1 function is evaluation at the nodes."""

    def __init__(self, qp, l, N_aux):
        super().__init__(qp)
        assert l is not None
        self._rows, self._l, self.m = qp.bc.free_dofs('fom'), l, N_aux
        self._xy_dev = None

    def _sample(self):
        # centres from numpy's global stream, in the reference's order (VirtualObservables.py:184-190) ...
        centres = np.array([[np.random.uniform(), np.random.uniform()] for _ in range(self.m)])
        device = self.qp._device
        if device is None or torch.device(device).type != "cuda":
            return fem.rbf_weighting(self.qp.physics.mesh, self._rows, centres, self._l)
        # ... evaluated at the fine free nodes on the device (resample() runs at every VO update)
        return self._evaluate_on_device(centres, device)

    def _evaluate_on_device(self, centres, device):
        """V [..., d, m] of centres [..., m, 2]."""
        if self._xy_dev is None:
            self._xy_dev = _as_f64(self.qp.physics.mesh.coords[self._rows], device)
        c = _as_f64(centres, device)
        d2 = (self._xy_dev[:, None, :] - c[..., None, :, :]).pow(2).sum(-1)
        return torch.exp(-d2 / self._l ** 2)

    def sample_V_batch(self, count):
        # one vector draw: numpy's legacy RandomState yields the same doubles as the 2 m count scalar draws of count
        # sample_V() calls, in the same order
        centres = np.random.uniform(size=(count, self.m, 2))
        device = self.qp._device
        if device is None or torch.device(device).type != "cuda":
            return np.stack([fem.rbf_weighting(self.qp.physics.mesh, self._rows, c, self._l) for c in centres])
        return self._evaluate_on_device(centres, device)


class GaussianSketchingSampler(BaseSampler):
    """i.i.d. N(0,1) weighting vectors (VirtualObservables.py:230-258)."""

    def __init__(self, qp, N_aux):
        super().__init__(qp)
        self.m = N_aux

    def _sample(self):
        device = self.qp._device
        if device is None or torch.device(device).type != "cuda":
            return np.stack([np.random.normal(0, 1, self.qp.dim_out) for _ in range(self.m)], axis=1)
        # drawn on the device (resample() runs at every VO update: no host loop, no H2D copy of d x m doubles); the
        # device generator is seeded from numpy's global stream, so np.random.seed() still fixes the sequence
        gen = torch.Generator(device=device)
        gen.manual_seed(int(np.random.randint(0, 2 ** 31 - 1)))
        return torch.randn(self.qp.dim_out, self.m, generator=gen, dtype=_F64, device=device)


class CoarseGrainedResidualSampler(BaseSampler):
    """V = W, constant (VirtualObservables.py:297-321)."""

    is_constant = True

    def __init__(self, qp, W):
        super().__init__(qp)
        self._W = W          # numpy [d,n] or ONE float64 device tensor shared by the samplers of all data points
        self._cached = None
        self.m = int(W.shape[1])

    def _sample(self):
        return self._W

    def sample(self):
        if self._cached is None:   # dense (Gamma, alpha) only when somebody asks for them
            self._cached = self.qp.weak_galerkin_on_device(self._W)
        return self._cached


class ConcatenatedSamplers(BaseSampler):
    """Columns of several samplers side by side (VirtualObservables.py:260-294); one device pass."""

    def __init__(self, samplers):
        super().__init__(None)
        self._samplers = list(samplers)

    qp = property(lambda self: self._samplers[0].qp)
    m = property(lambda self: sum(s.m for s in self._samplers))
    is_constant = property(lambda self: all(s.is_constant for s in self._samplers))
    provides_V = property(lambda self: all(s.provides_V for s in self._samplers))
    precision_mask = property(lambda self: np.concatenate([s.precision_mask for s in self._samplers]))

    def sample(self):
        """(Gamma, alpha) of every member stacked (VirtualObservables.py:283-294).  Constant members (V = W, flux
        constraints) return their cached pair; the others share ONE pass of the residual kernels over their columns."""
        if any(isinstance(s, FluxConstrainSampler) for s in self._samplers) or any(s.is_constant for s in self._samplers):
            pairs = []
            fresh = [s for s in self._samplers if not s.is_constant]
            fresh_pair = None
            if fresh:
                Vs = [s.sample_V() for s in fresh]
                dev = next((p.device for p in Vs if isinstance(p, torch.Tensor)), None)
                V = torch.cat([_as_f64(p, dev) for p in Vs], dim=1) if dev is not None else np.hstack(Vs)
                fresh_pair = self.qp.weak_galerkin_on_device(V)
            lo = 0
            for s in self._samplers:
                if s.is_constant:
                    pairs.append(s.sample())
                else:
                    pairs.append((fresh_pair[0][lo:lo + s.m], fresh_pair[1][lo:lo + s.m]))
                    lo += s.m
            dev = pairs[0][0].device
            return (torch.cat([_as_f64(G, dev) for G, _ in pairs], dim=0),
                    torch.cat([_as_f64(al, dev).reshape(-1) for _, al in pairs], dim=0))
        return self.qp.weak_galerkin_on_device(self._sample())

    def _sample(self):
        parts = [s.sample_V() for s in self._samplers]
        if any(isinstance(p, torch.Tensor) for p in parts):
            dev = next(p.device for p in parts if isinstance(p, torch.Tensor))
            return torch.cat([_as_f64(p, dev) for p in parts], dim=1)
        return np.hstack(parts)


class FluxConstrainSampler(BaseSampler):
    """Flux-balance constraints of the coarse cells (VirtualObservables.py:323-349): the reduced (Gamma, alpha) of a
    FluxConstraintReducedOrderModel (gpde_b200/flux.py, the FEniCS-free bottleneck/flux.py:43-158) for this data point,
    constant, learnable precision.  ``precomputed`` = this data point's (Gamma [N,d], alpha [N]) out of a batched device
    assembly of the whole ensemble (QuerryEnsemble.FromQuerryPointEnsemble)."""

    is_constant = True
    provides_V = False

    def __init__(self, qp, FluxConstrain, precomputed=None):
        super().__init__(qp=qp)
        if not FluxConstrain.initialized:
            raise RuntimeError('Initialize flux-constrain first')
        if precomputed is not None:
            self._Gamma_fc, self._alpha_fc = precomputed
        else:
            self._Gamma_fc, self._alpha_fc = FluxConstrain.assemble_reduced(np.exp(qp.x), qp.bc)

    m = property(lambda self: int(self._alpha_fc.numel() if isinstance(self._alpha_fc, torch.Tensor) else np.asarray(self._alpha_fc).size))
    precision_mask = property(lambda self: np.ones(self.m))

    def sample(self):
        device = self.qp._device
        if device is None and torch.cuda.is_available():
            device = torch.device("cuda", torch.cuda.current_device())
        return _as_f64(self._Gamma_fc, device), _as_f64(self._alpha_fc, device).reshape(-1)

    def _sample(self):
        raise NotImplementedError


# ======================================================================================= linear query
class LinearQuerry(object):
    """Gamma [m,d], Gamma^T and alpha [m] of one data point as float64 device tensors (VirtualObservables.py:353-447).

    What is KEPT is the weighting matrix V [d,m] of the sampler; the dense Gamma = V^T K / alpha = V^T f are produced by the
    residual kernels the first time somebody reads them (the ensemble's batched update never does: it works on V)."""

    def __init__(self, querry_point, sampler, dtype, device):
        self._querry_point, self._sampler = querry_point, sampler
        self.dtype, self.device = dtype, device
        self._store = {}
        self._V = None
        self.resample(ForceResample=True)

    def _materialise(self):
        if "Gamma" not in self._store:
            if self._V is None:
                raise RuntimeError("LinearQuerry holds neither V nor (Gamma, alpha)")
            self._set(*self._querry_point.weak_galerkin_on_device(self._V, device=self.device))

    def _f64_slot(name):
        def get(self):
            self._materialise()
            return self._store.get(name)

        def put(self, value):
            assert value.dtype == torch.double
            self._store[name] = value
        return property(get, put)

    Gamma = _f64_slot("Gamma")
    GammaTransposed = _f64_slot("GammaTransposed")
    alpha = _f64_slot("alpha")
    del _f64_slot

    V = property(lambda self: self._V, doc="weighting matrix [d,m] (None for samplers that only provide Gamma, alpha)")
    m = property(lambda self: int(self._V.shape[1]) if self._V is not None else self.Gamma.shape[0],
                 doc="number of virtual observables")
    dim_out = property(lambda self: int(self._V.shape[0]) if self._V is not None else self.Gamma.shape[1])
    precision_mask = property(lambda self: self._sampler.precision_mask)

    def _set(self, Gamma, alpha):
        self._store["Gamma"] = _as_f64(Gamma, self.device)
        self._store["alpha"] = _as_f64(alpha, self.device)
        self._store["GammaTransposed"] = self._store["Gamma"].t()

    def resample(self, ForceResample=False):
        if ForceResample or not self._sampler.is_constant:
            self._store.clear()
            if getattr(self._sampler, "provides_V", True):
                self._V = _as_f64(self._sampler.sample_V(), self.device)
            else:
                self._V = None
                self._set(*self._sampler())

    def temporary_set_galerkin_manually(self, V):
        self._V = _as_f64(V, self.device)
        self._store.clear()
        self.precision = -torch.ones(self.m, dtype=torch.double, device=self.device)


class QuerryEnsemble(object):
    """VirtualObservables.py:450-543."""

    def __init__(self, querries, dtype, device):
        self._querries, self.dtype, self.device = list(querries), dtype, device

    def __len__(self):
        return len(self._querries)

    def __getitem__(self, item):
        return self._querries[item]

    def __iter__(self):
        return iter(self._querries)

    N = property(lambda self: len(self._querries))
    m = property(lambda self: sum(q.m for q in self._querries), doc="total number of pieces of information")
    precision_mask = property(lambda self: self._querries[0].precision_mask)
    dim_out = property(lambda self: self._querries[0].dim_out)

    def resample(self, ForceResample=False):
        for q in self._querries:
            q.resample(ForceResample=ForceResample)

    @classmethod
    def FromQuerryPointEnsemble(cls, QuerryPointEnsemble, physics, CGR, flux, N_gaussian, N_rbf, l_rbf=None, *,
                                dtype=None, device=None):
        assert isinstance(physics, dict) and dtype is not None and device is not None
        W = physics['W']
        if W is None:
            raise NotImplementedError('need to provide W (as numpy array)')
        assert isinstance(W, np.ndarray) and W.shape[0] > W.shape[1]
        if N_rbf > 0:
            assert l_rbf is not None
        querries = []
        W_dev = _as_f64(W, device)      # ONE device copy of W shared by the samplers of all data points
        flux_pairs = None
        if flux:
            # test functions of the coarse cells' flux balances (VirtualObservables.py:514-517): the sparse pattern once,
            # then (Gamma, alpha) of ALL data points in one device product instead of one FEniCS assembly per data point
            from .flux import FluxConstraintReducedOrderModel
            fluxconstr = FluxConstraintReducedOrderModel(physics)
            fluxconstr.create_measures()
            if torch.device(device).type == "cuda":
                a_all = torch.exp(_as_f64(np.stack([qp.x for qp in QuerryPointEnsemble]), device))
                flux_pairs = fluxconstr.assemble_reduced_batched(a_all, QuerryPointEnsemble.dirichlet_values(_F64, device), device)
        for n_qp, qp in enumerate(QuerryPointEnsemble):
            qp._device = device
            parts = []
            if CGR:
                parts.append(CoarseGrainedResidualSampler(qp, W_dev))
            if flux:
                parts.append(FluxConstrainSampler(qp, fluxconstr, precomputed=None if flux_pairs is None else
                                                  (flux_pairs[0][n_qp], flux_pairs[1][n_qp])))
            if N_gaussian > 0:
                parts.append(GaussianSketchingSampler(qp, N_gaussian))
            if N_rbf > 0:
                parts.append(RadialBasisFunctionSampler(qp, l_rbf, N_rbf))
            sampler = parts[0] if len(parts) == 1 else ConcatenatedSamplers(parts)
            querries.append(LinearQuerry(qp, sampler, dtype=dtype, device=device))
        return cls(querries, dtype=dtype, device=device)


# ======================================================================================= virtual observables
class BaseVirtualObservable(object):
    def __init__(self, querry_point, dtype, device):
        assert isinstance(querry_point, QuerryPoint)
        self._querry_point, self.dtype, self.device = querry_point, dtype, device

    querry_point = property(lambda self: self._querry_point)
    d_y = property(lambda self: self._querry_point.dim_out)


class VirtualObservable(BaseVirtualObservable):
    """Posterior N(mean, diag(vars)) of one data point's fine solution given its virtual observables
    (VirtualObservables.py:596-669)."""

    def __init__(self, querry, querry_point, dtype, device):
        super().__init__(querry_point, dtype, device)
        assert isinstance(querry, LinearQuerry)
        self._querry = querry
        self._mean = self._vars = self._noise = None
        # member of a VirtualObservablesEnsemble: its batched update keeps the posterior of ALL data points in two [N,d]
        # tensors; this object reads its row from there unless it has been updated on its own since (generation counter)
        self._ens, self._k, self._own_gen = None, -1, -1

    def _posterior_row(self, which):
        ens = self._ens
        if ens is not None and ens._post is not None and self._own_gen != ens._post_gen:
            return ens._post[which][self._k]
        return self._mean if which == 0 else self._vars

    querry = property(lambda self: self._querry)
    mean = property(lambda self: self._posterior_row(0))
    vars = property(lambda self: self._posterior_row(1))
    m = property(lambda self: self._querry.m)

    @property
    def vo_variances(self):
        return self._noise

    @vo_variances.setter
    def vo_variances(self, value):
        assert value.dtype == torch.double and value.device == self.device
        self._noise = value

    def resample(self, ForceResample=False):
        self._querry.resample(ForceResample=ForceResample)

    def _set_posterior(self, mean, vars_):
        self._mean, self._vars = mean, vars_
        if self._ens is not None:
            self._own_gen = self._ens._post_gen
            self._ens._members_dirty = True
            self._ens.flush_cache()

    @torch.no_grad()
    def update(self, g, prec, iteration, *, ForceUpdate=False):
        if not ForceUpdate:
            raise RuntimeError
        q = self._querry
        mean, vars_ = condition_gaussian(q.Gamma.unsqueeze(0), q.alpha.unsqueeze(0), self._noise,
                                         g.to(_F64).unsqueeze(0), prec.to(_F64).unsqueeze(0))
        self._set_posterior(mean[0], vars_[0])


class BaseVirtualObservablesEnsemble(object):
    """VirtualObservables.py:796-905."""

    def __init__(self, QuerryPointEnsemble, virtual_observables, dtype, device):
        self._QuerryPointEnsemble = QuerryPointEnsemble
        self._virtual_observables = list(virtual_observables)
        self.dtype, self.device = dtype, device
        assert all(vo.m == self._virtual_observables[0].m for vo in self._virtual_observables)
        self._cache = {}

    def __getitem__(self, item):
        return self._virtual_observables[item]

    def __iter__(self):
        return iter(self._virtual_observables)

    def __len__(self):
        return len(self._virtual_observables)

    X = property(lambda self: self._QuerryPointEnsemble.X)
    N = property(lambda self: len(self._virtual_observables))
    m = property(lambda self: self._virtual_observables[0].m)
    M = property(lambda self: sum(vo.m for vo in self._virtual_observables))
    dim_out = property(lambda self: self._virtual_observables[0].d_y)

    def flush_cache(self):
        self._cache.clear()

    def _stacked(self, what):
        if what not in self._cache:
            rows = [getattr(vo, what) for vo in self._virtual_observables]
            assert all(r.dtype == torch.double for r in rows)
            self._cache[what] = torch.stack(rows).to(device=self.device, dtype=self.dtype)
        return self._cache[what].detach()

    mean = property(lambda self: self._stacked("mean"))
    vars = property(lambda self: self._stacked("vars"))
    logsigma = property(lambda self: 0.5 * torch.log(self.vars))

    def update(self, G, PREC, iteration, writer=None):
        self.update_vo_precision(iteration, writer)
        for n, vo in enumerate(self._virtual_observables):
            vo.update(G[n, :], PREC[n, :], iteration, ForceUpdate=True)
        self.flush_cache()

    def update_vo_precision(self, iteration, writer=None):
        raise NotImplementedError

    def resample(self, ForceResample=False):
        for vo in self._virtual_observables:
            vo.resample(ForceResample=ForceResample)


class VirtualObservablesEnsemble(BaseVirtualObservablesEnsemble):
    """VirtualObservables.py:908-998 with every loop over the data points replaced by a launch over all of them:

      update               rho(G) -> gpde_vo_posterior_f64          (2 launches; the reference: N x [3 einsum + cholesky + ...])
      update_vo_precision  rho(mean) -> gpde_vo_moments_f64 -> sum  (2 launches + one [N,m] reduction)
      residuals            one residual launch

    all matrix-free on the samplers' weighting matrices V (no dense Gamma [N,m,d]).  Up to ``max_kernel_m`` = 64 virtual
    observables per data point the update is one posterior launch; up to ``max_blocked_m`` = 256 it is the blocked route
    (gpde_vo_posterior_blocked_f64: three launches, Lambda_n in a device workspace, data points chunked so that the
    workspace stays within ``max_stack_bytes``).  Ensembles that contain samplers without a weighting matrix (flux
    constraints) or more than 256 virtual observables per data point condition densely (``condition_gaussian``: torch /
    cuBLAS / cuSOLVER), chunked by ``max_stack_bytes``.  ``last_update_route`` says which route the last update took:
    "kernel", "blocked" or "dense"."""

    # per-chunk budget for the stacked Gamma [n,m,d] of the dense route and the workspace of the blocked route
    max_stack_bytes = 1 << 30
    max_kernel_m = 64
    max_blocked_m = 256

    def __init__(self, QuerryPointEnsemble, QuerryEnsemble, dtype, device):
        vos = [VirtualObservable(q, qp, dtype=dtype, device=device) for q, qp in zip(QuerryEnsemble, QuerryPointEnsemble)]
        super().__init__(QuerryPointEnsemble, vos, dtype=dtype, device=device)
        self._QuerryEnsemble = QuerryEnsemble
        self._alpha_0 = self._beta_0 = 1e-6
        self._prec_alpha = 0.5 * self.N + self._alpha_0
        self._prec_beta = torch.ones(self.m, dtype=torch.double, device=self.device)
        self._infinite_precision_mask = torch.tensor(QuerryEnsemble[0].precision_mask < 0, dtype=torch.bool,
                                                     device=self.device)
        self._mean_vo_variances = self._get_mean_vo_variances()
        self._set_member_variance_values(self._mean_vo_variances)
        self._precision_initialized = False
        self._resident = None
        self._post, self._post_gen, self._members_dirty = None, 0, False
        self._info = None
        self.last_update_route = None
        for k, vo in enumerate(self._virtual_observables):
            vo._ens, vo._k = self, k

    infinite_precision_mask = property(lambda self: self._infinite_precision_mask)
    fixed_precision = property(lambda self: bool(self._infinite_precision_mask.all().item()))

    def _get_mean_vo_variances(self):
        mv = self._prec_beta / (self._prec_alpha + 1)   # VirtualObservables.py:962-966
        mv[self._infinite_precision_mask] = 0
        return mv

    def _set_member_variance_values(self, mean_vo_vars):
        for vo in self._virtual_observables:
            vo._noise = mean_vo_vars

    def _stacked(self, what):
        # posterior of all data points straight from the batched update unless a member was updated on its own since
        if self._post is not None and not self._members_dirty and what in ("mean", "vars"):
            return self._post[0 if what == "mean" else 1].to(dtype=self.dtype).detach()
        return super()._stacked(what)

    # -- device-resident inputs of the whole ensemble -------------------------------------------
    def _inputs(self):
        """(plan, conductivities a[N,*], Dirichlet values g[N,n_bc]) of all data points, resident on the device.

        The fields of the data points never change, so exp(x) is taken ONCE here (the reference likewise evaluates
        np.exp(x) once per QuerryPoint when it assembles and caches K, VirtualObservables.py:52-59) and every
        residual launch runs with a_is_log = 0.  When the DG0 fields come from images (both cells of a pixel carry
        the same value, bottleneck/utils.py:123-129) the per-pixel layout and the structured-grid kernels are used."""
        if self._resident is None:
            qpe = self._QuerryPointEnsemble
            physics = qpe[0].physics
            X = np.stack([qp.x for qp in qpe])
            plan, field = None, X
            try:
                pix = physics.mesh.pixel_of_cell()
                img = np.empty((X.shape[0], physics.mesh.nx * physics.mesh.ny))
                img[:, pix] = X
                if np.array_equal(img[:, pix], X):
                    plan, field = VoPlan.cached(physics, self.device, pixel_input=True), img
            except Exception:   # noqa: BLE001 -- not a pixel mesh: per-cell input
                plan = None
            if plan is None:
                plan = VoPlan.cached(physics, self.device)
            a = torch.exp(_as_f64(field, self.device))
            self._resident = (plan, a, qpe.dirichlet_values(_F64, self.device))
        return self._resident

    def _weights(self, max_m=None):
        """Weighting matrices of the data points for the batched kernels: one shared [d,m] tensor (every LinearQuerry holds
        the SAME tensor: V = W of the coarse-grained-residual sampler) or the stack [N,d,m]; None when some data point has
        no weighting matrix or m exceeds ``max_m`` (default ``max_kernel_m``; dense route).  The stack is rebuilt after
        resample()."""
        Vs = [vo.querry.V for vo in self._virtual_observables]
        if any(v is None for v in Vs) or Vs[0].shape[1] > (self.max_kernel_m if max_m is None else max_m):
            return None
        if all(v is Vs[0] for v in Vs):
            return Vs[0]
        key = tuple((v.data_ptr(), v._version) for v in Vs)
        cached = getattr(self, "_stacked_V", None)
        if cached is None or cached[0] != key:
            cached = (key, Vs, torch.stack(Vs))        # (holds the members: their addresses cannot be recycled under the key)
            self._stacked_V = cached
        return cached[2]

    def _shared_weights(self, V, B):
        """V as the residual kernels take it.  A contiguous float64 tensor on this device is packed once and the packed
        copy reused while it stays the same tensor at the same version (V = W of the coarse-grained-residual sampler only
        changes at resample(), VirtualObservables.py:297-321); the cache holds a reference to exactly that tensor, so its
        address cannot be recycled under the key.  Anything else (numpy, other dtype / device, strided) is converted and
        packed inside the call, every call."""
        plan = self._inputs()[0]
        if not (isinstance(V, torch.Tensor) and V.dtype == _F64 and V.is_cuda and V.device == plan.device and V.is_contiguous()):
            return _as_f64(V, self.device)
        key = (V.data_ptr(), V._version, tuple(V.shape), int(B))
        cached = getattr(self, "_packed_weights", None)
        if cached is None or cached[0] != key or cached[1] is not V:
            cached = (key, V, plan.pack_weights(V, int(B)))
            self._packed_weights = cached
        return cached[2]

    def _own_weights(self):
        """The querries' own weighting matrices for residuals / residual_gradients without V: the shared [d,m] tensor or
        the stack [N,d,m]."""
        V = self._weights(max_m=float("inf"))
        if V is None:
            raise RuntimeError("residuals / residual_gradients without V need every data point's weighting matrix; some "
                             "sampler of this ensemble provides only (Gamma, alpha) (flux constraints): pass V explicitly")
        return V

    def residuals(self, Y, V=None):
        """r[N,m] = V_n^T (K_fom(x_n) y~_n - f) for all data points in one call.  V [d,m] is a weighting matrix shared by
        the ensemble (e.g. V = W of the coarse-grained-residual sampler); without V the querries' own weighting matrices
        are used (shared, or one per data point as with Gaussian-sketch and RBF samplers), so that r[n] = Gamma_n Y[n] -
        alpha_n."""
        plan, a, G = self._inputs()
        if V is None:
            V = self._own_weights()
        V = V if isinstance(V, torch.Tensor) and V.dim() == 3 else self._shared_weights(V, Y.shape[0])
        return plan.residual(a, _as_f64(Y, self.device), G, V, a_is_log=False)

    def residual_gradients(self, S, V=None):
        """q[N,d] = K_ff(x_n) V_n s_n = Gamma_n^T S[n] for all data points in one call (S [N,m]); V as for residuals."""
        plan, a, _ = self._inputs()
        if V is None:
            V = self._own_weights()
        return plan.residual_T(a, _as_f64(V, self.device), _as_f64(S, self.device), a_is_log=False)

    def _fine_residual(self, Y):
        """rho[N,d] = (K_fom(a_n) y~_n - f)_free of all data points: one rho-only residual launch."""
        plan, a, gbc = self._inputs()
        _, rho = plan.residual(a, Y, gbc, None, a_is_log=False)
        return rho

    def check(self):
        """Reads and clears the device info word of the batched update; raises if some Lambda_n was not positive definite
        (torch.cholesky raises at the same point of the reference, VirtualObservables.py:658)."""
        if self._info is not None:
            flag = int(self._info.item())
            if flag:
                self._info.zero_()
                raise RuntimeError("virtual-observable update: Lambda = Gamma C Gamma^T + Sigma is not positive definite")

    @torch.no_grad()
    def update(self, G, PREC, iteration, writer=None):
        self.update_vo_precision(iteration, writer)
        G64, P64 = _as_f64(G, self.device), _as_f64(PREC, self.device)
        V = self._weights(max(self.max_kernel_m, self.max_blocked_m))
        if V is not None:
            plan, a, _ = self._inputs()
            if self._info is None:
                self._info = torch.zeros(1, dtype=torch.int32, device=self.device)
            rho = self._fine_residual(G64)
            if self.m <= self.max_kernel_m:
                mean, vars_ = plan.posterior(a, V, rho, self._mean_vo_variances, G64, P64, info=self._info)
                self.last_update_route = "kernel"
            else:
                mean, vars_ = self._posterior_blocked(plan, a, V, rho, G64, P64)
                self.last_update_route = "blocked"
            self._post, self._members_dirty = (mean, vars_), False
            self._post_gen += 1
        else:
            self.last_update_route = "dense"
            vos = self._virtual_observables
            per = 8 * self.m * self.dim_out
            step = max(1, int(self.max_stack_bytes // max(per, 1)))
            self._post = None
            for lo in range(0, self.N, step):
                chunk = vos[lo:lo + step]
                Gam = torch.stack([vo.querry.Gamma for vo in chunk])
                alp = torch.stack([vo.querry.alpha for vo in chunk])
                mean, vars_ = condition_gaussian(Gam, alp, self._mean_vo_variances, G64[lo:lo + step], P64[lo:lo + step])
                for k, vo in enumerate(chunk):
                    vo._set_posterior(mean[k], vars_[k])
        self.flush_cache()

    def _posterior_blocked(self, plan, a, V, rho, G64, P64):
        """The blocked route over chunks of data points whose workspace fits ``max_stack_bytes``."""
        N = self.N
        per = max(1, plan.posterior_blocked_workspace_bytes(1, self.m))     # the most bytes per data point (most row segments)
        step = max(1, int(self.max_stack_bytes // per))
        if step >= N:
            return plan.posterior_blocked(a, V, rho, self._mean_vo_variances, G64, P64, info=self._info)
        mean, vars_ = torch.empty_like(G64), torch.empty_like(G64)
        for lo in range(0, N, step):
            sl = slice(lo, lo + step)
            mean[sl], vars_[sl] = plan.posterior_blocked(a[sl] if a.dim() == 2 else a, V[sl] if V.dim() == 3 else V, rho[sl],
                                                         self._mean_vo_variances, G64[sl], P64[sl], info=self._info)
        return mean, vars_

    @torch.no_grad()
    def update_vo_precision(self, iteration, writer=None):
        if not self._precision_initialized:
            self._precision_initialized = True
            return
        if self[0].mean is None or self[0].vars is None:
            raise RuntimeError
        if self.fixed_precision:
            return
        V = self._weights(max(self.max_kernel_m, self.max_blocked_m))
        if V is not None:     # VirtualObservables.py:985-990 for all data points: two launches and one reduction
            plan, a, _ = self._inputs()
            mean, vars_ = _as_f64(self._stacked("mean"), self.device), _as_f64(self._stacked("vars"), self.device)
            r, s2 = plan.moments(a, V, self._fine_residual(mean), vars_)
            beta = (r * r + s2).sum(dim=0)
        else:
            beta = torch.zeros(self.m, dtype=torch.double, device=self.device)
            for vo in self._virtual_observables:
                Gam = vo.querry.Gamma
                beta += (Gam @ vo.mean - vo.querry.alpha) ** 2 + (Gam ** 2) @ vo.vars
        self._prec_beta = 0.5 * beta + self._beta_0
        self._mean_vo_variances = self._get_mean_vo_variances()
        self._set_member_variance_values(self._mean_vo_variances)
        if writer is not None:
            writer.add_scalar('Monitor/Mean_VO_variances', torch.mean(self._mean_vo_variances), global_step=iteration)


# ======================================================================================= energy VO
class EnergyVirtualObservable(BaseVirtualObservable):
    """Energy-type virtual observable (VirtualObservables.py:672-788): subspace Newton steps on
    1/2 mu^T A mu - b^T mu with A = diag(prec) + K/T, b = f/T + prec*g,
        mean <- mean - V (V^T A V)^-1 V^T (A mean - b),   vars = 1 / (prec + diag(K)/T).
    The reference forms the dense d x d matrix A on the CPU; here K is never formed:
        A mean - b = prec*(mean - g) + rho(mean)/T      rho = K_ff mean - f_eff   (one residual launch)
        A V        = prec*V + (K_ff V)/T                K_ff V = residual_T with s = I, shared field
    and the m x m system is solved on the device.  diag(K) is taken once at construction from the host
    assembly, like the reference's ``self._querry_point.K.diagonal()`` (:701, setup time)."""

    def __init__(self, querry_point, num_iterations_per_update, stochastic_subspace=None, sampler=None, l=0.1,
                 dtype=None, device=None):
        if dtype is None or device is None:
            raise ValueError('need to provide dtype and device')
        super().__init__(querry_point, dtype=dtype, device=device)
        self._stochastic_subspace = stochastic_subspace
        self._num_iterations_per_update = num_iterations_per_update
        if sampler is None:
            if stochastic_subspace is None:
                raise ValueError
            sampler = RadialBasisFunctionSampler(self._querry_point, l=l, N_aux=stochastic_subspace)
        self._sampler = sampler
        self._temperature = 1
        self._temperature_schedule = None
        self._mean = self._vars = None
        self._forced_temperature = None
        self._K_diag = _as_f64(self._querry_point.K.diagonal(), self.device)      # setup time (:701)
        self._plan = VoPlan.cached(self._querry_point.physics, self.device)
        self._x = _as_f64(self._querry_point.x, self.device)
        self._g_bc = _as_f64(self._querry_point.dirichlet_values(), self.device)
        load = self._querry_point.bc.assemble_vanilla_force_vector(self._querry_point.physics.identifier)
        # the cached plan carries no load vector (zero for both reference factories): keep f_free separately
        self._load_free = _as_f64(load[self._querry_point.physics.free_dofs], self.device) if np.any(load != 0) else None

    @property
    def temperature(self):
        return self._temperature if self._forced_temperature is None else self._forced_temperature

    def force_temperature(self, value):
        self._forced_temperature = value

    mean = property(lambda self: self._mean)
    vars = property(lambda self: self._vars)
    m = property(lambda self: 1)

    def resample(self, ForceResample=False):
        pass   # nothing to be done (:726-728)

    def set_temperature(self, temperature):
        assert temperature >= 0
        self._temperature = temperature

    def set_temperature_schedule(self, type, T_init, T_final, num_steps):
        assert type.lower() in ['linear', 'exponential']
        cls = LinearTemperatureSchedule if type.lower() == 'linear' else ExponentialTemperatureSchedule
        self._temperature_schedule = cls(T_init, T_final, num_steps)

    def set_linear_temperature_schedule(self, T_init=1, T_final=0.0001, num_steps=None):
        if num_steps is None:
            raise ValueError
        self._temperature_schedule = LinearTemperatureSchedule(T_init, T_final, num_steps)

    def update_precision(self, iteration):
        if self._forced_temperature is not None:
            return
        if self._temperature_schedule is None:
            raise RuntimeError
        self._temperature = self._temperature_schedule.get_temperature(iteration)

    @torch.no_grad()
    def update(self, g, prec, iteration, *, ForceUpdate=False):
        if not ForceUpdate:
            raise RuntimeError
        inv_T = 1.0 / self.temperature
        prec = prec.detach().to(_F64).to(self.device)
        g = g.detach().to(_F64).to(self.device)
        self._vars = 1.0 / (prec + inv_T * self._K_diag)
        if self._mean is None:
            self._mean = torch.zeros(self.d_y, dtype=_F64, device=self.device)
        plan, x, gbc = self._plan, self._x, self._g_bc
        for _ in range(self._num_iterations_per_update):
            V = _as_f64(self._sampler.sample_V(), self.device)                        # [d, m]
            m = V.shape[1]
            eye = torch.eye(m, dtype=_F64, device=self.device)
            KV = plan.residual_T(x, V, eye)                                            # [m, d], rows (K_ff V e_j)^T
            M = V.t() @ (prec.unsqueeze(1) * V) + inv_T * (KV @ V)                    # V^T A V (K symmetric)
            _, rho = plan.residual(x, self._mean.unsqueeze(0), gbc, None)             # rho = K_ff mean - f_eff
            if self._load_free is not None:
                rho = rho - self._load_free
            grad = prec * (self._mean - g) + inv_T * rho[0]                            # A mean - b
            self._mean = self._mean - V @ torch.linalg.solve(M, V.t() @ grad)

    def __repr__(self):
        return 'Energy virtual Observable | Current temperature = {}'.format(self._temperature)


class _ReplaySampler(BaseSampler):
    """Hands out weighting matrices that were drawn earlier, in their order."""

    def __init__(self, qp, Vs):
        super().__init__(qp)
        self._Vs = iter(Vs)

    def _sample(self):
        return next(self._Vs)


class EnergyVirtualObservablesEnsemble(BaseVirtualObservablesEnsemble):
    """VirtualObservables.py:1001-1037 with the loop over the data points replaced by launches over all of them:

      update   per Newton iteration: rho(mean) of all data points (one residual launch) -> gpde_vo_energy_step_f64
               (one launch); the reference: N x n_it x [dense V^T A V, V^T (A mean - b), solve]

    The weighting matrices are drawn in the member loop's order (data point-major, iteration-minor), with one
    ``sample_V_batch`` call when the data points share one sampler, so both routes see the same draws.  Up to
    ``max_kernel_m`` = 64 weighting functions the step is gpde_vo_energy_step_f64; for ``max_kernel_m`` < m <=
    ``max_blocked_m`` it is the blocked gpde_vo_energy_step_blocked_f64 (three launches, M_n in a workspace).  The member
    loop (``EnergyVirtualObservable.update`` per data point) runs instead when ``batched_update`` is False, when the m
    announced by the samplers or drawn exceeds both limits, or when the members differ in iterations per update or
    physics; ``last_update_route`` says which route the last update took ("batched", "blocked" or "members")."""

    batched_update = True
    max_kernel_m = 64
    # the blocked route takes max_kernel_m < m <= max_blocked_m (at most 256, the kernels' limit); at 64 it is off and
    # such m take the member loop
    max_blocked_m = 64
    # per-chunk budget for the drawn weighting matrices V [n, n_it, d, m] (and the blocked route's workspace)
    max_stack_bytes = 1 << 30

    def __init__(self, QuerryPointEnsemble, num_iterations_per_update, sampler, dtype, device):
        vos = [EnergyVirtualObservable(qp, num_iterations_per_update, sampler=sampler, dtype=dtype, device=device)
               for qp in QuerryPointEnsemble]
        super().__init__(QuerryPointEnsemble, vos, dtype=dtype, device=device)
        self._resident = None
        self._info = None
        self.last_update_route = None

    def _inputs(self):
        """(plan, conductivities a [N,n_inputs], Dirichlet values [N,n_bc], diag(K) [N,d], free load [N,d] or None) of
        all data points, stacked once from the members: their fields, boundary data and diag(K) never change."""
        if self._resident is None:
            vos = self._virtual_observables
            loads = [vo._load_free for vo in vos]
            load = None
            if any(f is not None for f in loads):
                load = torch.stack([f if f is not None else torch.zeros_like(vo._K_diag) for f, vo in zip(loads, vos)])
            self._resident = (vos[0]._plan, torch.exp(torch.stack([vo._x for vo in vos])),
                              torch.stack([vo._g_bc for vo in vos]), torch.stack([vo._K_diag for vo in vos]), load)
        return self._resident

    def _draw(self, chunk, n_it):
        """V [n, n_it, d, m] of the data points of ``chunk`` in the member loop's order."""
        s = chunk[0]._sampler
        if all(vo._sampler is s for vo in chunk):
            V = _as_f64(s.sample_V_batch(len(chunk) * n_it), self.device)
        else:
            V = torch.cat([_as_f64(vo._sampler.sample_V_batch(n_it), self.device) for vo in chunk])
        return V.view(len(chunk), n_it, *V.shape[1:])

    def _update_members(self, G, PREC, iteration):
        for n, vo in enumerate(self._virtual_observables):
            vo.update(G[n, :], PREC[n, :], iteration, ForceUpdate=True)
        self.flush_cache()
        self.last_update_route = "members"

    @torch.no_grad()
    def update(self, G, PREC, iteration, writer=None):
        self.update_vo_precision(iteration, writer)
        vos = self._virtual_observables
        v0 = vos[0]
        n_it = v0._num_iterations_per_update
        m_known = [getattr(vo._sampler, "m", None) for vo in vos]
        max_m = max(self.max_kernel_m, self.max_blocked_m)
        if not self.batched_update or any(vo._num_iterations_per_update != n_it or vo._plan is not v0._plan for vo in vos) \
                or any(m is not None and m > max_m for m in m_known):
            return self._update_members(G, PREC, iteration)
        plan, a, gbc, K_diag, load = self._inputs()
        G64, P64 = _as_f64(G, self.device), _as_f64(PREC, self.device)
        inv_T = torch.tensor([1.0 / vo.temperature for vo in vos], dtype=_F64, device=self.device)
        vars_ = 1.0 / (P64 + inv_T.unsqueeze(1) * K_diag)           # the member's expression, row by row
        mean = torch.stack([vo._mean if vo._mean is not None else torch.zeros_like(vo._K_diag) for vo in vos])
        if self._info is None:
            self._info = torch.zeros(1, dtype=torch.int32, device=self.device)
        # m of samplers that do not announce it is known after the first draw: size the first chunk for the largest m
        # the batched routes take
        m = max((m for m in m_known if m is not None), default=max_m)
        route = "batched"
        lo = 0
        while lo < self.N:
            step = max(1, int(self.max_stack_bytes // self._chunk_bytes_per_point(plan, n_it, m)))
            chunk = vos[lo:lo + step]
            V = self._draw(chunk, n_it)
            m = int(V.shape[-1])
            if m > max_m:                  # only on the first chunk: the member loop, with the draws already made
                saved = [vo._sampler for vo in chunk]
                try:
                    for k, vo in enumerate(chunk):
                        vo._sampler = _ReplaySampler(vo.querry_point, V[k])
                    return self._update_members(G, PREC, iteration)
                finally:
                    for vo, s in zip(chunk, saved):
                        vo._sampler = s
            energy_step = plan.energy_step
            if m > self.max_kernel_m:
                energy_step, route = plan.energy_step_blocked, "blocked"
            hi = lo + len(chunk)
            V = V.transpose(0, 1).contiguous()                          # [n_it, n, d, m]: one contiguous stack per step
            for it in range(n_it):
                _, rho = plan.residual(a[lo:hi], mean[lo:hi], gbc[lo:hi], None, a_is_log=False)
                if load is not None:
                    rho -= load[lo:hi]
                energy_step(a[lo:hi], V[it], rho, G64[lo:hi], P64[lo:hi], inv_T[lo:hi], mean[lo:hi], info=self._info)
            lo = hi
        if int(self._info.item()):
            self._info.zero_()
            raise RuntimeError("energy virtual-observable update: V^T A V is not positive definite for some data point")
        for k, vo in enumerate(vos):
            vo._mean, vo._vars = mean[k], vars_[k]
        self.flush_cache()
        self.last_update_route = route

    def _chunk_bytes_per_point(self, plan, n_it, m):
        """Device bytes a data point adds to a chunk: its drawn V [n_it, d, m] and, on the blocked route, its workspace
        (sized for a chunk of one data point, which has the most row segments)."""
        ws = plan.posterior_blocked_workspace_bytes(1, m) if m > self.max_kernel_m else 0
        return 8 * n_it * self.dim_out * m + ws

    def force_temperature(self, value):
        for vo in self:
            vo.force_temperature(value)

    def set_temperature(self, *args, **kwargs):
        for vo in self:
            vo.set_temperature(*args, **kwargs)

    def set_temperature_schedule(self, type, **kwargs):
        for vo in self:
            vo.set_temperature_schedule(type, **kwargs)

    def set_linear_temperature_schedule(self, *args, **kwargs):
        for vo in self:
            vo.set_linear_temperature_schedule(*args, **kwargs)

    def update_vo_precision(self, iteration, writer=None):
        for vo in self._virtual_observables:
            vo.update_precision(iteration)
        if writer is not None:
            writer.add_scalar('Monitoring/Temperature', self._virtual_observables[0].temperature, global_step=iteration)


# ======================================================================================= schedules
class TemperatureSchedule(object):
    """T(iteration) between T_init and T_final over num_steps (VirtualObservables.py:1040-1091)."""

    def __init__(self, T_init, T_final, num_steps):
        assert num_steps > 1 and T_final < T_init
        self._T_init, self._T_final, self._num_steps = T_init, T_final, num_steps

    def _progress(self, iteration):
        if iteration > self._num_steps:
            raise RuntimeError
        return iteration / (self._num_steps - 1)

    def get_temperature(self, iteration):
        raise NotImplementedError


class LinearTemperatureSchedule(TemperatureSchedule):
    def get_temperature(self, iteration):
        return self._T_init + self._progress(iteration) * (self._T_final - self._T_init)


class ExponentialTemperatureSchedule(TemperatureSchedule):
    def get_temperature(self, iteration):
        return self._T_init * np.exp(np.log(self._T_final / self._T_init) * self._progress(iteration))

"""ORACLE (test infrastructure, not product code): CPU restatement of the reference's
coarse-grained model, the same torch ops in the same order.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs may
import this module.

Pinned against the reference itself: tests/golden/make_golden.py imports
the reference tree's bottleneck/ROM.py + components.py under stub ``dolfin`` (oracle/ref_shim.py)
and stores its outputs; tests/test_oracle_golden.py checks this restatement against them.
The constants fed to it (M, W, dof sets) come from oracle/fem_p1.py, whose FEniCS
boundary is "parity unpinned" (see its header).
"""
import numpy as np
import torch


def get_stiffness(M, x, bc_dofs, dirichlet=True):
    """K[n,n,B] = M @ x^T, Dirichlet rows -> identity rows (bottleneck/ROM.py:91-100)."""
    K = torch.matmul(M, x.t())
    if dirichlet:
        K[bc_dofs] = 0
        K[bc_dofs, bc_dofs] = 1
    return K


def rom_call(M, bc_dofs, X, F, return_stiffness=False):
    """u[B,n] = A(X)^-1 F  (bottleneck/ROM.py:65-88; torch.solve == batched LU, :59-62)."""
    if F.dim() < 3:
        F = F.unsqueeze(2)
    trunc = 1e-12
    if (X <= trunc).any().item():  # bottleneck/ROM.py:74-76
        raise ValueError('At least one of the conductivity values supplied to the ROM was smaller than {}'.format(trunc))
    K = get_stiffness(M, X, bc_dofs, True)
    y = torch.linalg.solve(K.permute(2, 0, 1), F).squeeze(2)
    if return_stiffness:
        return y, K
    return y


def operator_forward_mean(M, bc_dofs, W, effprop, F):
    """mu_y[B,d] = W @ rom(exp(effprop)+1e-8, F)  (bottleneck/components.py:296-302)."""
    return torch.einsum('sk,nk->ns', [W, rom_call(M, bc_dofs, torch.exp(effprop) + 1e-8, F)])


def rom_fwd_adjoint(M, bc_dofs, logX, F, gbar_u):
    """One 'CGM fwd+adjoint solve' per sample through autograd, exactly what the reference
    does implicitly (SURVEY.md section 8 a6): returns u, dL/dlogX, dL/dF for L = <gbar_u, u>."""
    logX = logX.detach().clone().requires_grad_(True)
    F = F.detach().clone().requires_grad_(True)
    u = rom_call(M, bc_dofs, torch.exp(logX) + 1e-8, F)
    u.backward(gbar_u)
    return u.detach(), logX.grad.detach(), F.grad.detach()


def rom_fwd_adjoint_closed_form(M, bc_dofs, free_dofs, logX, F, gbar_u):
    """Same quantities from the closed-form SPD statement (SURVEY.md section 3.4), numpy fp64,
    sample by sample -- an independent check of the autograd route above."""
    M = np.asarray(M); logX = np.asarray(logX); F = np.asarray(F); gbar = np.asarray(gbar_u)
    B, E = logX.shape
    n = M.shape[0]
    fr, bc = np.asarray(free_dofs), np.asarray(bc_dofs)
    u = np.zeros((B, n)); gX = np.zeros((B, E)); gF = np.zeros((B, n))
    for b in range(B):
        x = np.exp(logX[b]) + 1e-8
        K = M @ x
        Kff, Kfc = K[np.ix_(fr, fr)], K[np.ix_(fr, bc)]
        g = F[b, bc]
        u[b, bc] = g
        u[b, fr] = np.linalg.solve(Kff, F[b, fr] - Kfc @ g)
        lam = np.zeros(n)
        lam[fr] = np.linalg.solve(Kff, gbar[b, fr])
        lam[bc] = gbar[b, bc] - Kfc.T @ lam[fr]
        gF[b] = lam
        lam_f = np.zeros(n); lam_f[fr] = lam[fr]
        gx = -np.einsum('i,ije,j->e', lam_f, M, u[b])
        gX[b] = gx * np.exp(logX[b])
    return u, gX, gF


# ------------------------------------------------------------------ refined reference with per-entry bounds
EPS64 = 2.0 ** -53
_LD_OK = np.finfo(np.longdouble).eps <= 1e-18   # x86 80-bit or IEEE quad; else mpmath accumulates the residuals


def _ext_residual(M_nz, x, rows, rhs, v):
    """rhs - (K v)[rows] with K = sum_e M_e x_e, v [B,n] over all dofs, accumulated in extended precision.
    Returns (residual, |rhs| + (|M| x |v|)[rows] in float64)."""
    I, J, E, V, n = M_nz
    row_of = -np.ones(n, dtype=np.int64); row_of[rows] = np.arange(len(rows))
    sel = row_of[I] >= 0
    ri, cj, e, val = row_of[I[sel]], J[sel], E[sel], V[sel]
    scale = np.abs(rhs).astype(np.float64)
    np.add.at(scale, (slice(None), ri), np.abs(val)[None] * x[:, e] * np.abs(np.asarray(v, dtype=np.float64)[:, cj]))
    if _LD_OK:
        ld = np.longdouble
        r = np.asarray(rhs).astype(ld)
        np.subtract.at(r, (slice(None), ri), val.astype(ld)[None] * x[:, e].astype(ld) * np.asarray(v).astype(ld)[:, cj])
        return r, scale
    import mpmath
    mpmath.mp.dps = 40
    r = np.empty(rhs.shape, dtype=object)
    for b in range(rhs.shape[0]):
        acc = [mpmath.mpf(t) for t in np.asarray(rhs[b])]
        for k in range(len(val)):
            acc[ri[k]] -= mpmath.mpf(float(val[k])) * mpmath.mpf(float(x[b, e[k]])) * mpmath.mpf(v[b, cj[k]])
        r[b] = acc
    return r, scale


def _refined_solve(Kff, residual):
    """K_ff v = rhs: a float64 solve refined twice; residual(v) gives (rhs - K_ff v, scale) in extended precision
    (v = 0 for the first solve).  Returns v in float64 and max |residual| / scale after the refinement."""
    ext = np.longdouble if _LD_OK else object
    hi = np.zeros(Kff.shape[:2]).astype(ext)
    for _ in range(3):
        res, _ = residual(hi)
        hi = hi + np.linalg.solve(Kff, np.asarray(res, dtype=np.float64)[..., None])[..., 0].astype(ext)
    res, scale = residual(hi)
    res = np.abs(np.asarray(res, dtype=np.longdouble if _LD_OK else np.float64)).astype(np.float64)
    rel = float((res / np.maximum(scale, 1e-300)).max()) if res.size else 0.0
    return np.asarray(hi, dtype=np.float64), rel


def rom_reference(M, bc_dofs, X, F, gbar, x_is_log, u=None):
    """Reference of the coarse-grained model's forward and adjoint on exactly the inputs a kernel sees, with a
    per-entry rounding-error scale for each output.

    M [n,n,E], X [B,E], F [B,n], gbar [B,n] as float64 (float32 inputs: their rounded values).  x = exp(X) + 1e-8 when
    x_is_log (dx = exp(X)), else x = X (dx = 1).  u [B,n]: the u an adjoint call was given; None: the exact one.

    u_f and lambda_f come from a float64 solve refined twice with the residual in long double (mpmath where long
    double is no wider than double).  The scales follow Higham's backward error for Cholesky, |dK| <= c eps |R^T||R|
    (|R^T||R| = |L||D||L^T| bounds the fill-in, |K_ff| alone does not), plus the assembly A = |M| x:
        S_u   = |K_ff^-1| ((|R^T||R| + A_ff)|u_f| + |F_f| + A_fc|g|),   g = F_c
        S_lam = |K_ff^-1| ((|R^T||R| + A_ff)|lam_f| + |gbar_f|),   S_lam_c = |gbar_c| + A_fc^T (|lam_f| + S_lam)
        S_gX  = dx (|lam_f|^T |M_e| (|u| + S_u) + S_lam^T |M_e| |u|)      (S_u = 0 for a given u)
    A kernel is right when |out - ref| <= c eps64 S entry by entry with c = 4 (hbw + T + 4), T the most terms of one
    assembled entry (see ``bound_ratio``).  u_c = F_c with scale 0: it must be exact.
    Returns a dict of float64 arrays u, S_u, lam, S_lam, gX, S_gX, the ints c, hbw, T, and the relative residuals
    res_u, res_lam of the refined solves."""
    M = np.asarray(M, dtype=np.float64)
    X, F, gbar = (np.asarray(a, dtype=np.float64) for a in (X, F, gbar))
    n, _, Ecount = M.shape
    B = X.shape[0]
    is_bc = np.zeros(n, dtype=bool); is_bc[np.asarray(bc_dofs, dtype=np.int64)] = True
    fr, bc = np.flatnonzero(~is_bc), np.flatnonzero(is_bc)
    with np.errstate(over='ignore'):
        dx = np.exp(X) if x_is_log else np.ones_like(X)
        x = dx + 1e-8 if x_is_log else X
    I, J, E = np.nonzero(M)
    V = M[I, J, E]
    M_nz, MT_nz = (I, J, E, V, n), (J, I, E, V, n)
    K = np.zeros((B, n * n)); A = np.zeros((B, n * n))
    np.add.at(K, (slice(None), I * n + J), V[None] * x[:, E])
    np.add.at(A, (slice(None), I * n + J), np.abs(V)[None] * x[:, E])
    K, A = K.reshape(B, n, n), A.reshape(B, n, n)
    Kff, Aff, Afc = K[:, fr][:, :, fr], A[:, fr][:, :, fr], A[:, fr][:, :, bc]
    g = F[:, bc]
    ext = np.longdouble if _LD_OK else object

    def fwd_res(v):   # F_f - K_fc g - K_ff v
        full = np.zeros((B, n)).astype(ext); full[:, bc] = g; full[:, fr] = v
        return _ext_residual(M_nz, x, fr, F[:, fr], full)

    def adj_res(v):   # gbar_f - K_ff v   (K_ff^T: the kernels factor the symmetric band)
        full = np.zeros((B, n)).astype(ext); full[:, fr] = v
        return _ext_residual(MT_nz, x, fr, gbar[:, fr], full)

    u_f, res_u = _refined_solve(Kff, fwd_res)
    lam_f, res_lam = _refined_solve(Kff, adj_res)
    u_ref = F.copy(); u_ref[:, fr] = u_f
    lam = np.zeros((B, n)); lam[:, fr] = lam_f
    lf = np.zeros((B, n)); lf[:, fr] = lam_f
    lc, _ = _ext_residual(MT_nz, x, bc, gbar[:, bc], lf)     # lambda_c = gbar_c - K_fc^T lambda_f
    lam[:, bc] = np.asarray(lc, dtype=np.float64)

    L = np.linalg.cholesky(Kff)
    absRR = np.abs(L) @ np.abs(np.swapaxes(L, 1, 2))
    Kinv = np.abs(np.linalg.inv(Kff))
    mv = lambda Mat, v: np.einsum('bij,bj->bi', Mat, v)
    S_u = np.zeros((B, n))
    S_u[:, fr] = mv(Kinv, mv(absRR + Aff, np.abs(u_f)) + np.abs(F[:, fr]) + mv(Afc, np.abs(g)))
    S_lam = np.zeros((B, n))
    S_lf = mv(Kinv, mv(absRR + Aff, np.abs(lam_f)) + np.abs(gbar[:, fr]))
    S_lam[:, fr] = S_lf
    S_lam[:, bc] = np.abs(gbar[:, bc]) + np.einsum('bfc,bf->bc', Afc, np.abs(lam_f) + S_lf)

    u_g = u_ref if u is None else np.asarray(u, dtype=np.float64)
    Su_g = S_u if u is None else np.zeros((B, n))
    free_row = ~is_bc[I]
    gi, gj, ge, gv = I[free_row], J[free_row], E[free_row], V[free_row]
    ld = np.longdouble if _LD_OK else np.float64
    gX = np.zeros((B, Ecount), dtype=ld)
    np.add.at(gX, (slice(None), ge), -(gv.astype(ld)[None] * lam[:, gi].astype(ld) * u_g[:, gj].astype(ld)))
    gX = np.asarray(gX * dx.astype(ld), dtype=np.float64)
    S_gX = np.zeros((B, Ecount))
    np.add.at(S_gX, (slice(None), ge), np.abs(gv)[None] * (np.abs(lam[:, gi]) * (np.abs(u_g[:, gj]) + Su_g[:, gj])
                                                          + S_lam[:, gi] * np.abs(u_g[:, gj])))
    S_gX *= dx

    # half bandwidth of K_ff in free order and the most terms of one assembled entry
    fl = -np.ones(n, dtype=np.int64); fl[fr] = np.arange(len(fr))
    ff = (fl[I] >= 0) & (fl[J] >= 0)
    hbw = int(np.abs(fl[I[ff]] - fl[J[ff]]).max()) if ff.any() else 0
    T = int((M != 0).sum(axis=2).max())
    return dict(u=u_ref, S_u=S_u, lam=lam, S_lam=S_lam, gX=gX, S_gX=S_gX, c=4 * (hbw + T + 4), hbw=hbw, T=T,
                res_u=res_u, res_lam=res_lam)


def bound_ratio(out, ref, S, fp32=False):
    """max over entries of |out - ref| / (eps64 S + 2^-1074): the multiple of the rounding unit a kernel's error takes
    (compare with rom_reference's c).  A float32 output is first allowed its own rounding, 2^-24 |ref| + 2^-150 (half the
    smallest float32 subnormal); the 2^-1074 term is the absolute error of an operation in the float64 subnormal range."""
    out = np.asarray(out, dtype=np.float64); ref = np.asarray(ref, dtype=np.float64)
    if out.size == 0:
        return 0.0
    err = np.abs(out - ref)
    if fp32:
        err = np.maximum(err - (2.0 ** -24 * np.abs(ref) + 2.0 ** -150), 0.0)
    with np.errstate(invalid='ignore'):
        r = err / (EPS64 * np.asarray(S, dtype=np.float64) + 2.0 ** -1074)
    r[np.isnan(r)] = np.inf
    return float(r.max())

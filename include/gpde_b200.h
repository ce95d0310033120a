/*
 * gpde_b200.h -- C ABI of the B200-native physics layer (libgpde_b200.so).
 *
 * Drop-in boundary for the ONE hot path of pkmtum/generative-physics-informed-pde:
 *   - the coarse-grained model (assemble K(x)=sum_e x_e K_e, solve, adjoint):
 *       reference bottleneck/ROM.py:59-100  (+ autograd of it, SURVEY.md 8 a6)
 *       reference bottleneck/components.py:296-311 (exp(X)+1e-8, prolongation y = W u)
 *   - the virtual-observable residuals  r = V^T (K_fom(a) u~ - f)_free  and the transposed
 *     application  q = K_ff(a) (V s):
 *       reference bottleneck/VirtualObservables.py:57-69, 642-669, 971-998
 *
 * Conventions
 *   - plain C: pointers + sizes only, no torch / C++ types cross this boundary;
 *   - "host" pointers are read during the call and never retained;
 *   - "device" pointers must live on the plan's device; the library never allocates or frees
 *     user data -- scratch comes from the caller (query *_workspace_bytes first);
 *   - every launch goes to the caller's stream (a cudaStream_t passed as void*); no entry point
 *     synchronises the device except plan_create (uploads constants) and plan_destroy;
 *   - plans are immutable after creation => re-entrant across streams; one plan per device;
 *   - return value: 0 = ok, <0 = error (gpde_last_error() gives the text for this thread);
 *     numerical failures are reported LAPACK-style through a device info word, never by a trap;
 *   - matrices are row-major; batch is the leading axis (X[B,E], F[B,n], u[B,n], y[B,d] ...),
 *     exactly the torch layouts the reference passes around.
 *   - *_f64: double I/O.  *_f32: float I/O, double arithmetic inside (meets the 1e-5 tier).
 */
#ifndef GPDE_B200_H
#define GPDE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPDE_OK 0
#define GPDE_ERR_ARG (-1)      /* bad argument */
#define GPDE_ERR_CUDA (-2)     /* CUDA runtime error (allocation, launch) */
#define GPDE_ERR_SIZE (-3)     /* problem too large for this build's kernels */

/* info word bits written by the ROM kernels (atomicOr into *info, device int32) */
#define GPDE_INFO_NONPOSITIVE_X 1      /* some conductivity <= 1e-12   (ROM.py:74-76 -> ValueError) */
#define GPDE_INFO_NOT_SPD 2            /* non-positive pivot in the factorisation              */

typedef struct gpde_rom_plan gpde_rom_plan;
typedef struct gpde_vo_plan gpde_vo_plan;
typedef void *gpde_stream_t; /* cudaStream_t */

int gpde_version(void); /* 101: the residual family takes v_stride after V */
const char *gpde_last_error(void);

/* ------------------------------------------------------------------ coarse-grained model */

/* Replaces ROM.__init__ (bottleneck/ROM.py:8-15): keeps the element tensor and Dirichlet map on
 * the device, in the sparse/banded form the kernels use.
 *   M_host   [n,n,E] row-major, M[:,:,e] = unit-conductivity stiffness of coarse cell e (ROM.py:46-53)
 *   bc_dofs  [n_bc]  constrained dofs (physics.constrained_dofs, ROM.py:14)
 * Free dofs are the remaining ones, ascending and never reordered: the half bandwidth of K_ff is that of this order
 * (an unsorted or duplicated bc_dofs list gives the same plan).  Returns GPDE_ERR_ARG when no dof is free, and
 * GPDE_ERR_SIZE when the half bandwidth exceeds 255 or the cooperative kernels would need more than 227 KB of shared
 * memory per CTA: some meshes under ROM.FromPhysics's 290-cell cap are refused (the unit square with 36x4 or 52x1 cells
 * and left-right Dirichlet dofs; 51x1, half bandwidth 50, is accepted). */
int gpde_rom_plan_create(gpde_rom_plan **plan, int n, int E, const double *M_host,
                         const int64_t *bc_dofs, int n_bc, int device);
int gpde_rom_plan_destroy(gpde_rom_plan *plan);

/* out[0]=n, [1]=E, [2]=n_free, [3]=half bandwidth, [4]=factor doubles per sample,
 * [5]=assembly contributions, [6]=lanes per sample (1 = thread-per-sample kernels without a stash, 2 = windowed
 * thread-per-sample kernels: pass the stash to the forward call too, 8/16/32 = cooperative kernels), [7]=device */
int gpde_rom_plan_info(const gpde_rom_plan *plan, int64_t out[8]);

/* bytes of factor stash needed for a batch of B samples (always doubles; the layout is the kernels' business: the
 * windowed kernels interleave blocks of 128 samples, so size the buffer with this call, not with out[4] * B) */
size_t gpde_rom_factor_bytes(const gpde_rom_plan *plan, int64_t B);

/* Replaces ROM.__call__ (bottleneck/ROM.py:65-88)  [x_is_log = 0: X are conductivities]
 * and ReducedOrderModelOperator's exp(X)+1e-8 -> rom (components.py:298) [x_is_log = 1].
 *   X [B,E], F [B,n] (Dirichlet values already written at bc_dofs, BoundaryConditions.py:132-147)
 *   u [B,n]  solution incl. Dirichlet dofs
 *   factor   [gpde_rom_factor_bytes] banded LDL^T factor kept for the adjoint (may be NULL; plans with lanes == 2 then
 *            fall back to the slower cooperative kernels)
 *   info     device int32, OR-ed with GPDE_INFO_* (may be NULL)                              */
int gpde_rom_forward_f64(const gpde_rom_plan *plan, const double *X, int x_is_log, const double *F,
                         double *u, double *factor, int *info, int64_t B, gpde_stream_t stream);
int gpde_rom_forward_f32(const gpde_rom_plan *plan, const float *X, int x_is_log, const float *F,
                         float *u, double *factor, int *info, int64_t B, gpde_stream_t stream);

/* Replaces autograd through matmul/index_put/solve (SURVEY.md 3.4, 8 a6): with lambda = A^-T gbar_u,
 *   gradX[b,e] = - sum_{i free} sum_j lambda_i K_e[i,j] u_j   (times exp(X) when x_is_log)
 *   gradF[b,:] = lambda                                            (may be NULL)
 * factor == NULL => the factorisation is recomputed from X.                                  */
int gpde_rom_adjoint_f64(const gpde_rom_plan *plan, const double *X, int x_is_log, const double *u,
                         const double *factor, const double *gbar_u, double *gradX, double *gradF,
                         int64_t B, gpde_stream_t stream);
int gpde_rom_adjoint_f32(const gpde_rom_plan *plan, const float *X, int x_is_log, const float *u,
                         const double *factor, const float *gbar_u, float *gradX, float *gradF,
                         int64_t B, gpde_stream_t stream);

/* GetStiffness (bottleneck/ROM.py:91-100): K[n,n,B] (batch LAST, as the reference returns it),
 * Dirichlet rows replaced by identity rows when dirichlet != 0.  X are conductivities.       */
int gpde_rom_stiffness_f64(const gpde_rom_plan *plan, const double *X, double *K, int dirichlet,
                           int64_t B, gpde_stream_t stream);

/* Prolongation y = W u and its transpose gbar_u = W^T gbar_y (components.py:298 einsum 'sk,nk->ns')
 * with W[d,n] held as CSR on the device (rows have <= 3 non-zeros for P1).                    */
typedef struct gpde_prolong_plan gpde_prolong_plan;
int gpde_prolong_plan_create(gpde_prolong_plan **plan, int d, int n, const double *W_host, int device);
int gpde_prolong_plan_destroy(gpde_prolong_plan *plan);
int gpde_prolong_apply_f64(const gpde_prolong_plan *plan, const double *u, double *y, int64_t B,
                           gpde_stream_t stream);                 /* y[B,d]  = u[B,n] W^T */
int gpde_prolong_apply_T_f64(const gpde_prolong_plan *plan, const double *gy, double *gu, int64_t B,
                             gpde_stream_t stream);               /* gu[B,n] = gy[B,d] W   */
int gpde_prolong_apply_f32(const gpde_prolong_plan *plan, const float *u, float *y, int64_t B,
                           gpde_stream_t stream);
int gpde_prolong_apply_T_f32(const gpde_prolong_plan *plan, const float *gy, float *gu, int64_t B,
                             gpde_stream_t stream);

/* Fused operator epilogue (SURVEY.md section 8 row f1): the diagonal-Gaussian log-likelihood of the operator output
 * DiagonalGaussianLogLikelihood(Y, W u, 2 ls) (bottleneck/utils.py:231-241 on components.py:296-298, as evaluated at
 * generative.py:438-439) and its gradients, without writing mu_y = W u [B,d]:
 *     L  [B]   L_b   = -1/2 sum_i [2 ls_i + ((Y_bi - (W u_b)_i) / exp(ls_i))^2 + log 2 pi]        (always double)
 *     gu [B,n] dL_b/du_b = W^T ((Y_b - W u_b) exp(-2 ls))                          (may be NULL)
 *     gls[d]   d(sum_b L_b)/dls_i = sum_b (e_bi^2 - 1)                             (always double; may be NULL)
 * u [B,n], Y [B,d], ls [d] (log standard deviations, the operator's logsigmas_y).  L and gls are zeroed by the call, gls
 * also when B = 0.  The row kernel stages 32 samples of u in shared memory: n <= 799 coarse dofs, else GPDE_ERR_SIZE. */
int gpde_prolong_loglik_f64(const gpde_prolong_plan *plan, const double *u, const double *Y, const double *ls,
                            double *L, double *gu, double *gls, int64_t B, gpde_stream_t stream);
int gpde_prolong_loglik_f32(const gpde_prolong_plan *plan, const float *u, const float *Y, const float *ls,
                            double *L, float *gu, double *gls, int64_t B, gpde_stream_t stream);

/* Monte-Carlo predictive moments of the operator output per data point (generative.py:198-207: propagate_samples, then
 * torch.mean / torch.std over the S samples) without the [N S, d] samples: with ubar / Cov_u the sample mean / unbiased
 * covariance of the S coarse solutions u[n,s,:],
 *     y_mean[n,i] = W_i . ubar_n,     y_std[n,i] = sqrt(W_i Cov_u,n W_i^T + exp(2 ls_i))
 * (the reference's estimator with the output noise integrated out).  u [N,S,n_coarse], ls [d], y_mean / y_std [N,d].
 * S = 1 takes Cov_u as zero: y_std = exp(ls), where torch.std of one sample would give NaN.  ubar, Cov_u and the S
 * samples live in shared memory: 8 (n (n + 1) + S n) bytes <= 200 KB, i.e. S <= 998 on the 4x4 coarse mesh (n = 25) and
 * S <= 234 on the 8x8 one (n = 81); larger S returns GPDE_ERR_SIZE. */
int gpde_prolong_moments_f64(const gpde_prolong_plan *plan, const double *u, const double *ls, double *y_mean,
                             double *y_std, int64_t N, int S, gpde_stream_t stream);
int gpde_prolong_moments_f32(const gpde_prolong_plan *plan, const float *u, const float *ls, float *y_mean,
                             float *y_std, int64_t N, int S, gpde_stream_t stream);

/* ------------------------------------------------------------------ virtual observables */

/* Replaces QuerryPoint._assemble_system / LinearEllipticPhysics.assemble_system
 * (VirtualObservables.py:57-59, physics/LinearElliptic.py:137-159): the fine operator is kept
 * matrix-free as element data; K_fom(a) = sum_c a[cell_to_input[c]] * Ke[c].
 *   cell_dofs     [n_cells,3]   P1 connectivity
 *   Ke            [n_cells,3,3] unit-conductivity element stiffness
 *   cell_to_input [n_cells]     index of the per-sample conductivity entry used by cell c
 *                               (identity for DG0 input; pixel id for image input)
 *   free_dofs [d], bc_dofs [n_bc]; f_full [n_nodes] load vector or NULL (zero)               */
int gpde_vo_plan_create(gpde_vo_plan **plan, int n_nodes, int n_cells, const int32_t *cell_dofs,
                        const double *Ke, const int32_t *cell_to_input, int n_inputs,
                        const int64_t *free_dofs, int d, const int64_t *bc_dofs, int n_bc,
                        const double *f_full, int device);
int gpde_vo_plan_destroy(gpde_vo_plan *plan);
/* out[0]=n_nodes, [1]=n_cells, [2]=n_inputs, [3]=d, [4]=n_bc, [5]=slots per row, [6]=device */
int gpde_vo_plan_info(const gpde_vo_plan *plan, int64_t out[8]);

/* Which kernels serve gpde_vo_residual_* for m weighting functions and elem_bytes (8 = f64, 4 = f32) I/O:
 * 3 = structured pixel grid, m > 32: V packing + ONE kernel that produces the fine residual inside the FP64 tensor-core
 *     contraction (vo_gridgemm.cuh) + the reduction of its partial tiles (three launches),
 * 2 = structured-grid kernel (V packing launch + one fused launch), 1 = generic fused kernel (one launch),
 * 0 = version-1 kernels (generic matvec + V padding + tensor-core contraction; three launches).  Informational (launch counting, tests).
 * 2 and 3 need a pixel mesh of the lean grid kernel (nx in {16, 32, 64, 128}, even ny) without a load vector, and shared
 * memory for the decomposition at elem_bytes; the load vector is assumed subtracted.  Calls whose pointers are not 16-byte
 * aligned, that pass y = NULL or that ask for rho fall back from 2 to 1. */
int gpde_vo_plan_kernel_path(const gpde_vo_plan *plan, int m, int elem_bytes);

/* scratch bytes for any residual / residual_T / residual_grad call on B samples with m weighting functions, either
 * layout of V (v_stride = 0 or d*m) */
size_t gpde_vo_workspace_bytes(const gpde_vo_plan *plan, int64_t B, int m);

/* The residual family (gpde_vo_residual_*, gpde_vo_residual_T_*, gpde_vo_residual_grad_*) takes V row-major with
 * V_b = V + b*v_stride: v_stride = 0 shares one V [d,m] across the batch, v_stride = d*m gives one matrix per sample,
 * V [B,d,m]; any other value returns GPDE_ERR_ARG.  With one matrix per sample the fine residual comes from the rho-only
 * route of gpde_vo_residual_* (the kernel the plan picks for it), then one contraction kernel streams V_b once; the
 * transposed application and the gradient first form the FP64 rows V_b s_b in the workspace with one expansion kernel,
 * then run the K_ff application of gpde_vo_residual_T_* (strided-y marching kernel on pixel grids, generic matvec
 * otherwise) or the gradient kernels.  Any m >= 1; FP32 I/O reads V, rho and s as floats and accumulates in FP64 (rho
 * itself is held as floats); the workspace must be 16-byte aligned; sums run in a fixed order, so results are
 * deterministic.  B = 0 is a no-op in either layout.
 *
 * r[B,m] = V^T (K_fom(a_b) u~_b - f)_free ,  u~ = y on free dofs, g on constrained dofs
 *        = Gamma_b y_b - alpha_b   (VirtualObservables.py:61-69, 662, 990).
 *   a   [B or 1, n_inputs]  (a_stride = n_inputs, or 0 to share one field across the batch)
 *   a_is_log != 0: a holds log-conductivities (QuerryPoint.x), exp() applied inside
 *   y   [B,d]   (NULL = zeros);  g [B or 1, n_bc] with g_stride = n_bc or 0 (NULL = zeros)
 *   V   [d,m] or [B,d,m] (v_stride) weighting matrices (NULL with m=0 and v_stride=0: only rho is produced)
 *   rho [B,d] optional output of the fine residual itself (may be NULL)
 *   flags: bit0 = ignore the load vector f
 *          bit1 = `workspace` already holds V packed by gpde_vo_pack_weights_f64 (same plan, m, bit0):
 *                 the call skips its packing launch; it fails with GPDE_ERR_ARG instead of falling
 *                 back when the lean structured-grid kernel cannot serve it (V must still be passed);
 *                 packing is for a shared V only: bit1 with v_stride != 0 returns GPDE_ERR_ARG
 *          bits 8-15 = number of SMs to leave to kernels the caller runs beside this call on other streams
 *                 (the structured-grid kernel sizes its last wave for the remaining SMs; 0 = all SMs)
 *   workspace: >= gpde_vo_workspace_bytes(plan, B, m) when m > 0 (per-sample V: it holds rho [B,d] when the caller
 *                 passes no rho output) */
int gpde_vo_residual_f64(const gpde_vo_plan *plan, const double *a, int64_t a_stride, int a_is_log,
                         const double *y, const double *g, int64_t g_stride, const double *V, int64_t v_stride,
                         int m, double *r, double *rho, void *workspace, int flags, int64_t B,
                         gpde_stream_t stream);
int gpde_vo_residual_f32(const gpde_vo_plan *plan, const float *a, int64_t a_stride, int a_is_log,
                         const float *y, const float *g, int64_t g_stride, const float *V, int64_t v_stride,
                         int m, float *r, float *rho, void *workspace, int flags, int64_t B,
                         gpde_stream_t stream);

/* Packs V[d,m] once into `workspace` (>= gpde_vo_workspace_bytes(plan, B, m), 16-byte aligned) in the
 * fragment order of the structured-grid residual kernel, for callers whose weighting functions stay fixed
 * over many residual calls (the CoarseGrainedResidual sampler's V = W, VirtualObservables.py:297-321, changes
 * only at resample()).  Returns 0 when packed (pass flags bit1 to gpde_vo_residual_f64 with that workspace),
 * 1 when this plan / m has no packed layout (call residual without bit1), < 0 on error. */
int gpde_vo_pack_weights_f64(const gpde_vo_plan *plan, const double *V, int m, int flags, void *workspace,
                             gpde_stream_t stream);
/* the same for FP32 I/O calls (gpde_vo_residual_f32 with flags bit1); the packed copy holds doubles either way */
int gpde_vo_pack_weights_f32(const gpde_vo_plan *plan, const float *V, int m, int flags, void *workspace,
                             gpde_stream_t stream);

/* Batched Gaussian conditioning of all data points of a virtual-observable ensemble in ONE launch, matrix-free
 * (VirtualObservable.update, bottleneck/VirtualObservables.py:642-669, looped over the data points at :891-898):
 *     Lambda_n = Gamma_n C_n Gamma_n^T + diag(noise_var),  C_n = diag(1 / prec_n),  Gamma_n^T = K_ff(a_n) V_n
 *     mean_n   = g_n - C_n Gamma_n^T Lambda_n^-1 (Gamma_n g_n - alpha_n),   Gamma_n g_n - alpha_n = V_n^T rho_n
 *     vars_n   = diag(C_n) - diag(C_n Gamma_n^T Lambda_n^-1 Gamma_n C_n)
 * a [N, n_inputs] conductivities (NOT logs; a_stride = 0: one field shared by all data points); V [d,m] shared
 * (v_stride = 0) or [N,d,m] (v_stride = d*m); m <= 64; rho [N,d] = the fine residual K_fom(a_n) g~_n - f of the prior
 * mean (the rho output of gpde_vo_residual with y = g); noise_var [m]; g, prec, mean, vars [N,d].
 * info (device int32, may be NULL) receives GPDE_INFO_NOT_SPD if some Lambda_n has a non-positive pivot.           */
int gpde_vo_posterior_f64(const gpde_vo_plan *plan, const double *a, int64_t a_stride, const double *V,
                          int64_t v_stride, int m, const double *rho, const double *noise_var, const double *g,
                          const double *prec, double *mean, double *vars, int *info, int64_t N, gpde_stream_t stream);

/* The same conditioning for 1 <= m <= 256 (m > 256: GPDE_ERR_SIZE), blocked: Lambda_n and L_n^-1 (m x m, m padded to a
 * multiple of 64) live in the caller's workspace instead of shared memory.  Three launches: the Gram blocks of Lambda_n
 * over row tiles (DMMA), one Cholesky / triangular-inverse CTA per data point, and the mean / variance rows.  Arguments
 * as gpde_vo_posterior_f64, plus workspace (16-byte aligned, device) of workspace_bytes >=
 * gpde_vo_posterior_blocked_workspace_bytes(plan, N, m); a null, misaligned or smaller workspace returns GPDE_ERR_ARG.
 * N = 0 is a no-op.  Results are deterministic for a given (plan, N, m): the row split of the Gram pass depends on N. */
size_t gpde_vo_posterior_blocked_workspace_bytes(const gpde_vo_plan *plan, int64_t N, int m);
int gpde_vo_posterior_blocked_f64(const gpde_vo_plan *plan, const double *a, int64_t a_stride, const double *V,
                                  int64_t v_stride, int m, const double *rho, const double *noise_var, const double *g,
                                  const double *prec, double *mean, double *vars, int *info, void *workspace,
                                  size_t workspace_bytes, int64_t N, gpde_stream_t stream);

/* The two per-data-point terms of the precision hyper-update (VirtualObservablesEnsemble.update_vo_precision,
 * bottleneck/VirtualObservables.py:985-990), all data points at once:
 *     out_r [n,j] = (V_n^T rho_n)_j          = (Gamma_n mean_n - alpha_n)_j  for rho_n = rho(mean_n)
 *     out_s2[n,j] = sum_i Gamma_n[j,i]^2 v[n,i]
 * m <= 256 (else GPDE_ERR_SIZE); m > 64 runs one CTA per (64-column panel, data point).                           */
int gpde_vo_moments_f64(const gpde_vo_plan *plan, const double *a, int64_t a_stride, const double *V, int64_t v_stride,
                        int m, const double *rho, const double *v, double *out_r, double *out_s2, int64_t N,
                        gpde_stream_t stream);

/* One subspace-Newton step of the energy-type virtual observables for all data points in ONE launch, matrix-free
 * (EnergyVirtualObservable.update, bottleneck/VirtualObservables.py:769-788, looped over the data points at :1001-1037):
 *     M_n    = V_n^T diag(prec_n) V_n + inv_T[n] V_n^T K_ff(a_n) V_n        (= V_n^T A_n V_n, A_n = diag(prec_n) + K/T_n)
 *     b_n    = V_n^T (prec_n (mean_n - g_n) + inv_T[n] rho_n)                (= V_n^T (A_n mean_n - b))
 *     mean_n = mean_n - V_n M_n^-1 b_n                                       (Cholesky of M_n, in place on mean)
 * a [N, n_inputs] conductivities (NOT logs; a_stride = 0: one field shared by all data points, else n_inputs); V [d,m]
 * shared (v_stride = 0) or [N,d,m] (v_stride = d*m); m <= 64 (else GPDE_ERR_SIZE); rho [N,d] = K_ff(a_n) mean_n - f_eff
 * (the rho output of gpde_vo_residual with y = mean, minus a load vector the plan does not carry); g, prec, mean [N,d];
 * inv_T [N] device doubles.  N = 0 is a no-op.
 * info (device int32, may be NULL) receives GPDE_INFO_NOT_SPD if some M_n has a non-positive pivot; that data point's mean
 * is left unchanged.                                                                                                   */
int gpde_vo_energy_step_f64(const gpde_vo_plan *plan, const double *a, int64_t a_stride, const double *V,
                            int64_t v_stride, int m, const double *rho, const double *g, const double *prec,
                            const double *inv_T, double *mean, int *info, int64_t N, gpde_stream_t stream);

/* The same step for 1 <= m <= 256 (m > 256: GPDE_ERR_SIZE), blocked: M_n (m x m, m padded to a multiple of 64) lives in
 * the caller's workspace instead of shared memory.  Three launches: the Gram blocks of M_n and b_n over row tiles (DMMA),
 * one Cholesky CTA per data point (the blocked posterior's factor kernel, no noise term), and mean_n -= V_n sol_n on the
 * rows of V_n.  Arguments as gpde_vo_energy_step_f64, plus workspace (16-byte aligned, device) of workspace_bytes >=
 * gpde_vo_posterior_blocked_workspace_bytes(plan, N, m): the layout is the blocked posterior's.  m <= 0, an a_stride
 * other than 0 or n_inputs, a v_stride other than 0 or d*m, a null operand, or a null, misaligned or smaller workspace
 * returns GPDE_ERR_ARG.  N = 0 is a no-op.  A data point whose M_n has a non-positive pivot ORs GPDE_INFO_NOT_SPD into
 * info and keeps its mean bitwise.  Results are deterministic for a given (plan, N, m): the row split of the Gram pass
 * depends on N.                                                                                                        */
int gpde_vo_energy_step_blocked_f64(const gpde_vo_plan *plan, const double *a, int64_t a_stride, const double *V,
                                    int64_t v_stride, int m, const double *rho, const double *g, const double *prec,
                                    const double *inv_T, double *mean, int *info, void *workspace,
                                    size_t workspace_bytes, int64_t N, gpde_stream_t stream);

/* q[B,d] = K_ff(a_b) (V_b s_b) = Gamma_b^T s_b  (VirtualObservables.py:663; with s = P r it is the
 * gradient of 1/2 r^T P r w.r.t. y).  With B = m, s = I, a_stride = 0 and a shared V it yields Gamma itself.
 * On the reference's pixel meshes with m <= 32 and a shared V this is one kernel (after a small packing launch of V^T):
 * the rows of V s are produced inside the marching kernel and never reach global memory; `workspace` holds the packed
 * V^T (or, on the other routes, V s [B,d]): >= gpde_vo_workspace_bytes(plan, B, m), 16-byte aligned.  V, v_stride as
 * for gpde_vo_residual_*. */
int gpde_vo_residual_T_f64(const gpde_vo_plan *plan, const double *a, int64_t a_stride, int a_is_log,
                           const double *V, int64_t v_stride, int m, const double *s, double *q, void *workspace,
                           int64_t B, gpde_stream_t stream);
int gpde_vo_residual_T_f32(const gpde_vo_plan *plan, const float *a, int64_t a_stride, int a_is_log,
                           const float *V, int64_t v_stride, int m, const float *s, float *q, void *workspace,
                           int64_t B, gpde_stream_t stream);

/* Gradient of r = gpde_vo_residual_*(a, y, g, V) with respect to the conductivity input and the Dirichlet values, for
 * an incoming gradient gbar_r [B,m].  With w~_b = V_b gbar_r_b on the free dofs and 0 on the Dirichlet dofs, and since
 * K(a) = sum_c a[cell_to_input[c]] K_c is linear in a:
 *     grad_a[b,p] = sum_{c : cell_to_input[c] = p} w~_b[c]^T K_c u~_b[c]     ([c] = the three dofs of cell c)
 *     grad_g[b,k] = (K_cf(a_b) w~_b)_k                                       (the Dirichlet rows of K(a) applied to w~)
 * a_is_log != 0: a holds x with a = exp(x) (no offset), and grad_a is the gradient in x: exp(x) times the above.
 * The load vector does not enter either gradient.  Arguments as for gpde_vo_residual_*: a [B or 1, n_inputs]
 * (a_stride = n_inputs or 0), y [B,d] (NULL = zeros), g [B or 1, n_bc] (g_stride = n_bc or 0, NULL = zeros), V and
 * v_stride.  Outputs are per sample even when a_stride or g_stride is 0: grad_a [B,n_inputs], grad_g [B,n_bc]; either
 * may be NULL.  workspace: >= gpde_vo_workspace_bytes(plan, B, m), 16-byte aligned (it holds w = gbar_r V^T in FP64;
 * FP32 I/O computes in FP64 too).  B = 0 is a no-op.  m <= 0, a NULL gbar_r, V or a, a bad stride or a NULL or
 * misaligned workspace return GPDE_ERR_ARG.  Every output is written by one thread in a fixed order: results are
 * deterministic. */
int gpde_vo_residual_grad_f64(const gpde_vo_plan *plan, const double *a, int64_t a_stride, int a_is_log,
                              const double *y, const double *g, int64_t g_stride, const double *V, int64_t v_stride,
                              int m, const double *gbar_r, double *grad_a, double *grad_g, void *workspace,
                              int64_t B, gpde_stream_t stream);
int gpde_vo_residual_grad_f32(const gpde_vo_plan *plan, const float *a, int64_t a_stride, int a_is_log,
                              const float *y, const float *g, int64_t g_stride, const float *V, int64_t v_stride,
                              int m, const float *gbar_r, float *grad_a, float *grad_g, void *workspace,
                              int64_t B, gpde_stream_t stream);

/* ---- fine-mesh label solves: batched preconditioned CG (setup-time replacement of the per-sample FEniCS / spsolve calls
 * of physics/LinearElliptic.py:85-101, 120-133 in utils/data.py:96-99).  One iteration = one gpde_vo_residual_f64 call with
 * y = p (rho output, flags bit0, no Dirichlet data: rho = K_ff(a) p for the whole batch) + one gpde_cg_step_f64 call.
 * All arrays device, float64: rhs, Ax, x, r, p [B,d]; dinv [B or 1, d] (dinv_stride = d or 0) the inverse diagonal of
 * K_ff(a_b); rz, stop2, rnorm2 [B] per-sample scalars owned by the caller.
 *   init: r = rhs - Ax (Ax = NULL: x0 = 0), p = dinv r, rz = r.p, rnorm2 = r.r, stop2 = tol^2 rhs.rhs
 *   step: alpha = rz / p.Ap; x += alpha p; r -= alpha Ap; z = dinv r; beta = r.z / rz; p = z + beta p; rz, rnorm2 updated;
 *         samples with rnorm2 <= stop2 are frozen. */
int gpde_cg_init_f64(const double *rhs, const double *Ax, const double *dinv, int64_t dinv_stride, double *r,
                     double *p, double *rz, double *stop2, double *rnorm2, double tol, int d, int64_t B,
                     int device, gpde_stream_t stream);
int gpde_cg_step_f64(const double *Ap, const double *dinv, int64_t dinv_stride, double *x, double *r, double *p,
                     double *rz, const double *stop2, double *rnorm2, int d, int64_t B, int device,
                     gpde_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GPDE_B200_H */

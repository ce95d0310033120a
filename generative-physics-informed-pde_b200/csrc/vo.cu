// Virtual-observable residuals on sm_100a, matrix-free.
//   r_b = V^T (K_fom(a_b) u~_b - f)_free          (= Gamma_b y_b - alpha_b,  VirtualObservables.py:61-69, 662)
//   q_b = K_ff(a_b) (V s_b)                        (= Gamma_b^T s_b,          VirtualObservables.py:663)
// The reference materialises K_fom as scipy CSR per data point with FEniCS and forms the dense
// Gamma = V^T K on the CPU; here K_fom(a) = sum_c a_c K_c is never formed: each free row i gathers its
// incident cells ("row-cell ELL", slot-major so that consecutive rows read consecutive words):
//   rho_i = sum_slots a[in] * (c0 * u_i + c1 * u~[j1] + c2 * u~[j2]) - f_i
//
// Kernel families, chosen per call (gpde_vo_plan_kernel_path):
//   vo_grid2.cuh     the reference's pixel meshes (verified at plan creation), FP32/FP64 I/O: marching flux-form kernel
//                    with the contraction on the FP64 tensor pipe inside the kernel (m <= 32), or producing rho for ...
//   vo_gridgemm.cuh  ... one kernel that also contracts rho with many weighting functions (m > 32), or for ...
//   vo_gemm.cuh      ... the FP64 tensor-core contraction rho[B,d] V[d,m];
//   vo_fused.cuh     any P1 diffusion mesh, m <= 32: edge-form matvec + ring-staged tiles + DMMA contraction;
//   version 1        (below) any mesh, any m, FP32/FP64: row-cell ELL matvec, then vo_gemm.cuh.
#include "common.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <type_traits>

namespace gpde {

struct VoDev {
    int n_nodes, n_cells, n_inputs, d, n_bc, nslots;
    const int *ell_in;    // [nslots*d] conductivity input index of the slot's cell
    const int *ell_j1;    // [nslots*d] source of the 2nd vertex: >=0 -> y index, <0 -> -(g index)-1
    const int *ell_j2;    // [nslots*d]
    const double *ell_c0, *ell_c1, *ell_c2;   // [nslots*d]
    const double *f_free;  // [d]
};

}  // namespace gpde

namespace gpde {

__device__ __forceinline__ double ldd(const double *p) { return *p; }
__device__ __forceinline__ double ldd(const float *p) { return (double)*p; }

constexpr int kVoThreads = 256;

}  // namespace gpde

#include "vo_fused.cuh"
#include "vo_grid2.cuh"
#include "vo_expand.cuh"
#include "vo_gemm.cuh"
#include "vo_gridgemm.cuh"
#include "vo_posterior.cuh"
#include "vo_posterior_blocked.cuh"
#include "vo_energy_blocked.cuh"
#include "vo_energy.cuh"
#include "vo_grad.cuh"
#include "vo_vb.cuh"

namespace gpde {
// A pixel mesh the structured-grid kernels (vo_grid2.cuh) serve, verified by build_grid_plan.
struct GridDev {
    int ok;
    int nx, ny;          // pixels per row, pixel rows; nodes are (nx+1) x (ny+1)
    int ncol;            // free node columns per row (nx - 1)
    long long in0, sy;   // conductivity entry of pixel (cx, cy) = in0 + cy * sy + cx
    double rh, scale;    // rh = chs / cvs, scale = cvs
    int has_load;
};

// Experiment switches (A/B runs of the kernel families).  Read from the environment ONCE per plan, in gpde_vo_plan_create,
// never on a launch path.
struct VoEnv {
    bool path_v1 = false;     // GPDE_VO_PATH=v1: version-1 kernels only
    bool path_fused = false;  // GPDE_VO_PATH=fused: no structured-grid kernels
    bool sync_staging = false;   // GPDE_VO_SYNC_STAGING
    int gemm_splits = 0;         // GPDE_GEMM_SPLITS: parts of the contraction length (0 = automatic)
    int grid2_split = 1;         // GPDE_GRID2_SPLIT: 0 = never cut the node rows over a cluster, 1 = automatic, n > 1 = force n
    bool gridgemm = true;        // GPDE_VO_GRIDGEMM=0: rho through HBM + vo_gemm_kernel instead of the one-kernel route (m > 32)
    bool fused_t = true;         // GPDE_VO_FUSED_T=0: residual_T as expansion kernel + marching kernel (w [B,d] through HBM)
    int grid2_spc = 0;           // GPDE_GRID2_SPC: samples per CTA of the lean grid kernel (0 = automatic, see grid2_samples_per_cta)
    VoEnv() {
        const char *e;
        if ((e = getenv("GPDE_VO_PATH"))) { path_v1 = strcmp(e, "v1") == 0; path_fused = strcmp(e, "fused") == 0; }
        sync_staging = getenv("GPDE_VO_SYNC_STAGING") != nullptr;
        if ((e = getenv("GPDE_GEMM_SPLITS"))) gemm_splits = std::max(0, std::min(8, atoi(e)));
        if ((e = getenv("GPDE_GRID2_SPLIT"))) grid2_split = std::max(0, std::min(8, atoi(e)));
        if ((e = getenv("GPDE_VO_GRIDGEMM"))) gridgemm = atoi(e) != 0;
        if ((e = getenv("GPDE_GRID2_SPC"))) grid2_spc = std::max(0, atoi(e));
        if ((e = getenv("GPDE_VO_FUSED_T"))) fused_t = atoi(e) != 0;
    }
};
}  // namespace gpde

struct gpde_vo_plan {
    gpde::VoDev dev;
    gpde::VoTiles tiles;
    gpde::GridDev grid;
    gpde::VoCsrDev csr;     // K_ff as CSR term lists (vo_posterior.cuh)
    gpde::VoGradDev grad;   // input -> cells lists and the Dirichlet rows of K (vo_grad.cuh)
    size_t fused_smem;
    int device;
    int n_sm;
    gpde::VoEnv env;
    std::vector<void *> allocs;
};

namespace gpde {

// rho[b,i] for S samples per CTA.  ea (shared) = conductivities of the S samples, exp() applied.
template <typename Ta, typename Ty, typename To, int S>
__global__ void __launch_bounds__(kVoThreads)
vo_matvec_kernel(VoDev P, const Ta *__restrict__ a, long long a_stride, int a_is_log,
                 const Ty *__restrict__ y, const Ta *__restrict__ g, long long g_stride, int sub_f,
                 double *__restrict__ rho_ws, int ws_stride, To *__restrict__ rho_out, long long B, int stage_a) {
    extern __shared__ double ea[];   // [S][n_inputs] when stage_a
    const int d = P.d;
    for (long long b0 = (long long)blockIdx.x * S; b0 < B; b0 += (long long)gridDim.x * S) {
        if (stage_a) {
            __syncthreads();
#pragma unroll
            for (int s = 0; s < S; ++s) {
                const long long b = min(b0 + s, B - 1);
                for (int p = threadIdx.x; p < P.n_inputs; p += kVoThreads) {
                    double v = ldd(a + b * a_stride + p);
                    ea[s * P.n_inputs + p] = a_is_log ? exp(v) : v;
                }
            }
            __syncthreads();
        }
        for (int i = threadIdx.x; i < d; i += kVoThreads) {
            double acc[S], yi[S];
#pragma unroll
            for (int s = 0; s < S; ++s) {
                const long long b = min(b0 + s, B - 1);
                yi[s] = y ? ldd(y + b * d + i) : 0.0;
                acc[s] = sub_f ? -P.f_free[i] : 0.0;
            }
            for (int t = 0; t < P.nslots; ++t) {
                const int k = t * d + i;
                const int in = P.ell_in[k], j1 = P.ell_j1[k], j2 = P.ell_j2[k];
                const double c0 = P.ell_c0[k], c1 = P.ell_c1[k], c2 = P.ell_c2[k];
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    const long long b = min(b0 + s, B - 1);
                    double av;
                    if (stage_a) av = ea[s * P.n_inputs + in];
                    else {
                        av = ldd(a + b * a_stride + in);
                        if (a_is_log) av = exp(av);
                    }
                    double u1, u2;
                    if (j1 >= 0) u1 = y ? ldd(y + b * d + j1) : 0.0;
                    else u1 = g ? ldd(g + b * g_stride + (-j1 - 1)) : 0.0;
                    if (j2 >= 0) u2 = y ? ldd(y + b * d + j2) : 0.0;
                    else u2 = g ? ldd(g + b * g_stride + (-j2 - 1)) : 0.0;
                    acc[s] = fma(av, fma(c0, yi[s], fma(c1, u1, c2 * u2)), acc[s]);
                }
            }
#pragma unroll
            for (int s = 0; s < S; ++s) {
                const long long b = b0 + s;
                if (b < B) {
                    if (rho_ws) rho_ws[b * ws_stride + i] = acc[s];
                    if (rho_out) rho_out[b * d + i] = (To)acc[s];
                }
            }
        }
        if (rho_ws)   // zero the K padding the tensor-core contraction reads
            for (int i = d + threadIdx.x; i < ws_stride; i += kVoThreads)
#pragma unroll
                for (int s = 0; s < S; ++s)
                    if (b0 + s < B) rho_ws[(b0 + s) * ws_stride + i] = 0.0;
    }
}

// w[B,d] = s[B,m] V^T
template <typename Tv>
__global__ void vo_expand_kernel(const Tv *__restrict__ s, const Tv *__restrict__ V, double *__restrict__ w,
                                 long long B, int d, int m) {
    const long long total = B * (long long)d;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / d;
        const int i = (int)(idx - b * d);
        double acc = 0.0;
        for (int q = 0; q < m; ++q) acc = fma(ldd(s + b * m + q), ldd(V + (long long)i * m + q), acc);
        w[idx] = acc;
    }
}

template <typename T>
static cudaError_t track_vo(gpde_vo_plan *pl, const T **dst, const std::vector<T> &src) {
    T *p = nullptr;
    cudaError_t e = upload(&p, src);
    if (p) pl->allocs.push_back((void *)p);
    *dst = p;
    return e;
}

// Edge form + tile staging lists for the fused kernels.  Leaves pl->tiles.ok = 0 when the mesh does not
// qualify (element matrices without zero row sums, an edge shared by more than two cells, or rings that
// would not fit in shared memory); the version-1 kernels then serve every call.
static cudaError_t build_fused_tiles(gpde_vo_plan *pl, int n_nodes, int n_cells, const int32_t *cell_dofs,
                                     const double *Ke, const int32_t *cell_to_input, int d,
                                     const std::vector<int> &src, const std::vector<double> &pl_f_free) {
    VoTiles &Tl = pl->tiles;
    memset(&Tl, 0, sizeof(Tl));
    pl->fused_smem = 0;
    double kmax = 0.0;
    for (size_t k = 0; k < (size_t)n_cells * 9; ++k) kmax = std::max(kmax, fabs(Ke[k]));
    for (int c = 0; c < n_cells; ++c)
        for (int l = 0; l < 3; ++l)
            if (fabs(Ke[9 * c + 3 * l] + Ke[9 * c + 3 * l + 1] + Ke[9 * c + 3 * l + 2]) > 1e-13 * kmax)
                return cudaSuccess;   // not a pure diffusion operator
    struct Nb { int node, in0, in1, ncell; double s0, s1; };
    std::vector<std::vector<Nb>> nbs(d);
    for (int c = 0; c < n_cells; ++c)
        for (int l = 0; l < 3; ++l) {
            const int v = cell_dofs[3 * c + l];
            if (src[v] < 0) continue;
            std::vector<Nb> &list = nbs[src[v]];
            for (int l2 = 0; l2 < 3; ++l2) {
                if (l2 == l) continue;
                const double coef = Ke[9 * c + 3 * l + l2];
                if (coef == 0.0) continue;
                const int w = cell_dofs[3 * c + l2];
                Nb *hit = nullptr;
                for (Nb &nb : list)
                    if (nb.node == w) hit = &nb;
                if (!hit) {
                    list.push_back(Nb{w, cell_to_input[c], cell_to_input[c], 1, coef, 0.0});
                } else if (hit->ncell == 1) {
                    hit->in1 = cell_to_input[c];
                    hit->s1 = coef;
                    hit->ncell = 2;
                } else {
                    return cudaSuccess;   // edge shared by > 2 cells
                }
            }
        }
    int nnb = 1;
    for (int i = 0; i < d; ++i) nnb = std::max(nnb, (int)nbs[i].size());
    const int nt = (d + kFR - 1) / kFR;
    // u ring holds y by free index; a ring holds the conductivity inputs
    std::vector<int> ulo(nt, INT32_MAX), uhi(nt, -1), alo(nt, INT32_MAX), ahi(nt, -1);
    for (int i = 0; i < d; ++i) {
        const int t = i / kFR;
        ulo[t] = std::min(ulo[t], i);
        uhi[t] = std::max(uhi[t], i + 1);
        for (const Nb &nb : nbs[i]) {
            if (src[nb.node] >= 0) {
                ulo[t] = std::min(ulo[t], src[nb.node]);
                uhi[t] = std::max(uhi[t], src[nb.node] + 1);
            }
            alo[t] = std::min(alo[t], std::min(nb.in0, nb.in1));
            ahi[t] = std::max(ahi[t], std::max(nb.in0, nb.in1) + 1);
        }
    }
    for (int t = 0; t < nt; ++t)
        if (ahi[t] < 0) { alo[t] = 0; ahi[t] = 1; }   // a tile of isolated rows
    RangeRing ru = build_ring(ulo, uhi), ra = build_ring(alo, ahi);
    const int n_bc = pl->dev.n_bc;
    const int block_bytes = nnb * kFR * 32 + kFR * 8;
    const int g_base = ru.ring * kPitchB;
    const int a_base = g_base + n_bc * kPitchB;
    const int rs_base = a_base + ra.ring * kPitchB;
    const int rec_base = rs_base + (int)sizeof(double) * kFS * kRhoPitch;
    const int meta_base = rec_base + block_bytes;
    const size_t smem = (size_t)meta_base + (size_t)nt * sizeof(TileMeta);
    if (smem > 110 * 1024) return cudaSuccess;   // keep two CTAs per SM; otherwise fall back
    std::vector<TileMeta> meta(nt);
    std::vector<char> blocks((size_t)nt * block_bytes, 0);
    for (int t = 0; t < nt; ++t) {
        meta[t] = TileMeta{ru.first[t], ru.count[t], ru.off[t], ra.first[t], ra.count[t], ra.off[t], 0, 0};
        char *blk = blocks.data() + (size_t)t * block_bytes;
        int4 *ro = reinterpret_cast<int4 *>(blk);
        double2 *rc = reinterpret_cast<double2 *>(blk + (size_t)nnb * kFR * 16);
        double *fo = reinterpret_cast<double *>(blk + (size_t)nnb * kFR * 32);
        for (int k = 0; k < kFR; ++k) {
            const int i = t * kFR + k;
            if (i >= d) {   // rows past the end: harmless offsets, zero coefficients
                for (int s = 0; s < nnb; ++s) {
                    ro[s * kFR + k] = make_int4(0, a_base, a_base, 0);
                    rc[s * kFR + k] = make_double2(0.0, 0.0);
                }
                fo[k] = 0.0;
                continue;
            }
            const int own = ru.offset_of(t, i) * kPitchB;
            const int pad_in = nbs[i].empty() ? alo[t] : nbs[i][0].in0;
            for (int s = 0; s < nnb; ++s) {
                if (s < (int)nbs[i].size()) {
                    const Nb &nb = nbs[i][s];
                    const int sj = src[nb.node];
                    const int ou = sj >= 0 ? ru.offset_of(t, sj) * kPitchB : g_base + (-sj - 1) * kPitchB;
                    ro[s * kFR + k] = make_int4(ou, a_base + ra.offset_of(t, nb.in0) * kPitchB,
                                                a_base + ra.offset_of(t, nb.in1) * kPitchB, own);
                    rc[s * kFR + k] = make_double2(nb.s0, nb.s1);
                } else {   // padding: zero conductance to itself
                    const int oa = a_base + ra.offset_of(t, pad_in) * kPitchB;
                    ro[s * kFR + k] = make_int4(own, oa, oa, own);
                    rc[s * kFR + k] = make_double2(0.0, 0.0);
                }
            }
            fo[k] = pl_f_free[i];
        }
    }
    Tl.n_tiles = nt; Tl.nnb = nnb; Tl.ring_u = ru.ring; Tl.ring_a = ra.ring; Tl.n_bc = n_bc;
    Tl.g_base = g_base; Tl.a_base = a_base; Tl.rs_base = rs_base;
    Tl.rec_base = rec_base; Tl.meta_base = meta_base; Tl.block_bytes = block_bytes;
    Tl.async_ok = (ru.mode != 0 && ra.mode != 0) ? 1 : 0;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = track_vo(pl, &Tl.meta, meta);
    if (e == cudaSuccess) e = track_vo(pl, &Tl.blocks, blocks);
    if (e == cudaSuccess) {
        pl->fused_smem = smem;
        Tl.ok = 1;
    }
    return e;
}


// Rows of K(a) over the free columns as CSR with, per stored entry, the list of (conductivity input, element-matrix entry)
// terms: K_ij(a) = sum_t a[term_in[t]] * term_coef[t].  row_of[node] = the node's row (< 0: not a row).  The free rows
// (K_ff) serve the batched posterior update (vo_posterior.cuh), the Dirichlet rows (K_cf) the gradient in g (vo_grad.cuh).
static cudaError_t build_csr_terms(gpde_vo_plan *pl, VoCsrDev &C, int d, const std::vector<int> &row_of, int n_cells,
                                   const int32_t *cell_dofs, const double *Ke, const int32_t *cell_to_input,
                                   const std::vector<int> &src) {
    struct Term { int in; double coef; };
    std::vector<std::vector<std::pair<int, std::vector<Term>>>> rows(d);
    for (int c = 0; c < n_cells; ++c)
        for (int l = 0; l < 3; ++l) {
            const int i = row_of[cell_dofs[3 * c + l]];
            if (i < 0) continue;
            for (int l2 = 0; l2 < 3; ++l2) {
                const int j = src[cell_dofs[3 * c + l2]];
                const double v = Ke[9 * c + 3 * l + l2];
                if (j < 0 || v == 0.0) continue;
                std::vector<Term> *hit = nullptr;
                for (auto &e : rows[i])
                    if (e.first == j) hit = &e.second;
                if (!hit) {
                    rows[i].push_back({j, {}});
                    hit = &rows[i].back().second;
                }
                hit->push_back(Term{cell_to_input[c], v});
            }
        }
    std::vector<int> row_ptr(d + 1, 0), col, term_ptr(1, 0), term_in;
    std::vector<double> term_coef;
    int max_row = 1;
    for (int i = 0; i < d; ++i) {
        std::sort(rows[i].begin(), rows[i].end(), [](const auto &x, const auto &y) { return x.first < y.first; });
        for (auto &e : rows[i]) {
            col.push_back(e.first);
            for (const Term &t : e.second) {
                term_in.push_back(t.in);
                term_coef.push_back(t.coef);
            }
            term_ptr.push_back((int)term_in.size());
        }
        row_ptr[i + 1] = (int)col.size();
        max_row = std::max(max_row, row_ptr[i + 1] - row_ptr[i]);
    }
    C.d = d; C.nnz = (int)col.size(); C.max_row = max_row;
    cudaError_t e = track_vo(pl, &C.row_ptr, row_ptr);
    if (e == cudaSuccess) e = track_vo(pl, &C.col, col);
    if (e == cudaSuccess) e = track_vo(pl, &C.term_ptr, term_ptr);
    if (e == cudaSuccess) e = track_vo(pl, &C.term_in, term_in);
    if (e == cudaSuccess) e = track_vo(pl, &C.term_coef, term_coef);
    return e;
}

// The cells of every conductivity input, ascending, with their dof sources and element matrices (vo_grad_cells_kernel).
static cudaError_t build_grad_cells(gpde_vo_plan *pl, int n_cells, const int32_t *cell_dofs, const double *Ke,
                                    const int32_t *cell_to_input, int n_inputs, const std::vector<int> &src) {
    std::vector<int> in_ptr(n_inputs + 1, 0);
    for (int c = 0; c < n_cells; ++c) in_ptr[cell_to_input[c] + 1]++;
    for (int p = 0; p < n_inputs; ++p) in_ptr[p + 1] += in_ptr[p];
    std::vector<int> next(in_ptr.begin(), in_ptr.end() - 1);
    std::vector<int4> cell_src(n_cells);
    std::vector<double> cell_K((size_t)n_cells * 9);
    for (int c = 0; c < n_cells; ++c) {
        const int e = next[cell_to_input[c]]++;
        cell_src[e] = make_int4(src[cell_dofs[3 * c]], src[cell_dofs[3 * c + 1]], src[cell_dofs[3 * c + 2]], 0);
        for (int k = 0; k < 9; ++k) cell_K[(size_t)e * 9 + k] = Ke[(size_t)c * 9 + k];
    }
    VoGradDev &G = pl->grad;
    G.n_inputs = n_inputs;
    cudaError_t e = track_vo(pl, &G.in_ptr, in_ptr);
    if (e == cudaSuccess) e = track_vo(pl, &G.cell_src, cell_src);
    if (e == cudaSuccess) e = track_vo(pl, &G.cell_K, cell_K);
    return e;
}

// Structured-grid detection for vo_grid2.cuh.  Leaves pl->grid.ok = 0 unless the element data is exactly the
// 5-point pixel operator the grid kernel evaluates on a mesh it is built for (every check below is against the
// arrays the caller passed, nothing is assumed from names):
//   nodes (nx+1) x (ny+1) numbered x-fastest, nx in {16, 32, 64, 128}, ny even; Dirichlet dofs = the columns ix = 0
//   and ix = nx, listed row by row (left, right); free dofs = all other nodes ascending; two cells per pixel sharing
//   one input entry in0 + cy*sy + cx; horizontal / vertical couplings uniform (chs / cvs), hypotenuse couplings zero.
static void build_grid_plan(gpde_vo_plan *pl, int n_nodes, int n_cells, const int32_t *cell_dofs, const double *Ke,
                            const int32_t *cell_to_input, int n_inputs, const int64_t *free_dofs, int d,
                            const int64_t *bc_dofs, int n_bc, const std::vector<double> &f_free) {
    GridDev &G = pl->grid;
    memset(&G, 0, sizeof(G));
    if (n_bc < 4 || (n_bc & 1) || bc_dofs[0] != 0) return;
    const long long nxn = bc_dofs[1] + 1;               // nodes per row
    if (nxn < 3 || n_nodes % nxn != 0) return;
    const int nx = (int)nxn - 1, nyn = (int)(n_nodes / nxn), ny = nyn - 1, ncol = nx - 1;
    if (ny < 1 || n_bc != 2 * nyn || d != ncol * nyn || n_cells != 2 * nx * ny || n_inputs != nx * ny) return;
    if (!(nx == 16 || nx == 32 || nx == 64 || nx == 128) || ny < 2 || (ny & 1)) return;
    for (int r = 0; r < nyn; ++r)
        if (bc_dofs[2 * r] != (long long)r * nxn || bc_dofs[2 * r + 1] != (long long)r * nxn + nx) return;
    for (int i = 0; i < d; ++i)
        if (free_dofs[i] != (long long)(i / ncol) * nxn + 1 + i % ncol) return;
    double kmax = 0.0;
    for (size_t k = 0; k < (size_t)n_cells * 9; ++k) kmax = std::max(kmax, fabs(Ke[k]));
    if (!(kmax > 0.0)) return;
    const double tol = 1e-13 * kmax;
    std::vector<int> sq_input((size_t)nx * ny, -1), sq_count((size_t)nx * ny, 0);
    // side coverage per square: bottom, top (horizontal), left, right (vertical)
    std::vector<unsigned char> side((size_t)nx * ny * 4, 0);
    double chs = 0.0, cvs = 0.0;
    bool have_h = false, have_v = false;
    for (int c = 0; c < n_cells; ++c) {
        int ix[3], iy[3];
        for (int l = 0; l < 3; ++l) {
            ix[l] = cell_dofs[3 * c + l] % (int)nxn;
            iy[l] = cell_dofs[3 * c + l] / (int)nxn;
        }
        const int cx = std::min(ix[0], std::min(ix[1], ix[2])), cy = std::min(iy[0], std::min(iy[1], iy[2]));
        if (cx >= nx || cy >= ny) return;
        for (int l = 0; l < 3; ++l)
            if (ix[l] - cx > 1 || iy[l] - cy > 1) return;
        const size_t sq = (size_t)cy * nx + cx;
        if (sq_count[sq] == 0) sq_input[sq] = cell_to_input[c];
        else if (sq_input[sq] != cell_to_input[c]) return;   // per-cell input: generic kernels
        if (++sq_count[sq] > 2) return;
        for (int l = 0; l < 3; ++l) {
            double rs = 0.0;
            for (int l2 = 0; l2 < 3; ++l2) rs += Ke[9 * c + 3 * l + l2];
            if (fabs(rs) > tol) return;                     // not a pure diffusion operator
            for (int l2 = 0; l2 < 3; ++l2) {
                if (l2 == l) continue;
                const double v = Ke[9 * c + 3 * l + l2];
                if (fabs(v - Ke[9 * c + 3 * l2 + l]) > tol) return;
                const int dx = ix[l2] - ix[l], dy = iy[l2] - iy[l];
                if (dx != 0 && dy != 0) {
                    if (fabs(v) > tol) return;               // hypotenuse must not couple
                } else if (dy == 0) {
                    if (!have_h) { chs = v; have_h = true; }
                    if (fabs(v - chs) > tol) return;
                    if (l < l2) side[sq * 4 + (iy[l] == cy ? 0 : 1)]++;
                } else {
                    if (!have_v) { cvs = v; have_v = true; }
                    if (fabs(v - cvs) > tol) return;
                    if (l < l2) side[sq * 4 + 2 + (ix[l] == cx ? 0 : 1)]++;
                }
            }
        }
    }
    if (!have_h || !have_v || chs == 0.0 || cvs == 0.0) return;
    for (size_t k = 0; k < side.size(); ++k)
        if (side[k] != 1) return;                          // every pixel side carried by exactly one cell
    for (size_t sq = 0; sq < sq_count.size(); ++sq)
        if (sq_count[sq] != 2) return;
    const long long in0 = sq_input[0];
    const long long sy = ny > 1 ? (long long)sq_input[nx] - in0 : nx;
    if (sy != nx && sy != -nx) return;
    for (int cy = 0; cy < ny; ++cy)
        for (int cx = 0; cx < nx; ++cx)
            if (sq_input[(size_t)cy * nx + cx] != in0 + cy * sy + cx) return;
    if ((in0 & 1) || (sy & 1)) return;

    G.nx = nx; G.ny = ny; G.ncol = ncol;
    G.in0 = in0; G.sy = sy; G.rh = chs / cvs; G.scale = cvs;
    G.has_load = 0;
    for (int i = 0; i < d; ++i)
        if (f_free[i] != 0.0) G.has_load = 1;
    G.ok = 1;
}

// GPDE_VO_PATH=v1 forces the unfused version-1 kernels (A/B testing, fallback check)
static bool use_fused(const gpde_vo_plan *pl) {
    return pl->tiles.ok && !pl->env.path_v1;
}

// GPDE_VO_PATH=fused keeps the structured-grid kernel out as well (generic fused kernel instead)
static bool use_grid(const gpde_vo_plan *pl) {
    return pl->grid.ok && !pl->env.path_v1 && !pl->env.path_fused;
}

// Bytes of one packed V row of the lean grid kernel: NT n-tiles and NX DFMA columns per strip, then the strips' masks.
static inline int grid2_v_row_bytes(int nstrips, int NT, int NX) {
    return nstrips * (4 * NT * 32 * 8 + NX * 128) + kGrid2MaskBytes;
}

// The decomposition of the lean grid kernel (vo_grid2.cuh) for m weighting functions (rho: no V inside); false when it
// does not apply (no pixel mesh, a load vector to subtract, m > 32, shared memory).
static bool grid2_setup(const gpde_vo_plan *pl, int m, bool rho, int sub_f, Grid2Dev &G, int &NT, int &NX, size_t &smem,
                        int ea = 8, int ey = 8) {   // ea / ey: bytes per element of a / y (8 or 4)
    const GridDev &G0 = pl->grid;
    const int nx = G0.nx, ny = G0.ny;
    if (!G0.ok) return false;
    if (G0.has_load && sub_f) return false;
    NT = 1; NX = 0;
    if (!rho) {
        if (m < 1 || m > 32) return false;
        NT = m >> 3; NX = m & 7;
        if (NX > 1 || NT == 0) { NT += NX ? 1 : 0; NX = 0; }
    }
    memset(&G, 0, sizeof(G));
    G.nx = nx; G.ny = ny; G.ncol = G0.ncol;
    for (G.lognx = 0; (1 << G.lognx) < nx; ++G.lognx) {}
    G.nstrips = nx / 16;
    for (G.lognstrips = 0; (1 << G.lognstrips) < G.nstrips; ++G.lognstrips) {}
    G.groups = 16 / G.nstrips;
    G.in0 = G0.in0; G.sy = G0.sy; G.rh = G0.rh; G.scale = G0.scale;
    const int S = 8 * G.groups;
    // pitches in elements, chosen against bank conflicts of the warp's reads (vo_grid2.cuh): FP32 rows need a_pitch = 16 mod 32
    // (LDS.128 of two samples per phase) and y_pitch = 4 mod 8 (the samples' phases then spread the banks)
    G.a_pitch = ea == 8 ? 2 * nx + 2 : 2 * nx + 16;
    G.y_pitch = ey == 8 ? 2 * nx + 8 : 2 * nx + 12;
    G.y_off = S * G.a_pitch * ea;
    G.v_off = 0;
    G.v_row_bytes = rho ? 0 : grid2_v_row_bytes(G.nstrips, NT, NX);
    G.stage_bytes = (G.y_off + S * G.y_pitch * ey + 127) & ~127;
    const size_t fixed = 2 * (size_t)G.stage_bytes + (4 * 16 + 8) * sizeof(unsigned long long) + 258 * sizeof(double);
    // V ring: three 2-row stages when they fit (the sample groups of a CTA may then drift a stage apart), else two
    G.nvs = rho ? 0 : ((fixed + 3 * 2 * (size_t)G.v_row_bytes <= 227 * 1024) ? 3 : 2);
    smem = fixed + (size_t)G.nvs * 2 * G.v_row_bytes;
    if (smem > 227 * 1024) return false;
    G.spc = S;
    return true;
}

// The lean grid kernel stages a in 16-byte pieces: base, sample stride and the plan's pixel offsets must be aligned.
static bool grid2_a_aligned(const gpde_vo_plan *pl, const void *a, long long a_stride, int ea) {
    return !((uintptr_t)a & 15) && !((a_stride * ea) & 15) && !((pl->grid.in0 * ea) & 15) && !((pl->grid.sy * ea) & 15);
}

// Samples per CTA of the lean grid kernel.  A CTA holds S = 8 * groups sample slots and owns a whole SM; with
// ceil(B / S) CTAs the last wave leaves SMs idle (4096 samples, S = 32: 128 CTAs on 148 SMs).  The kernel is bound by
// the bytes an SM streams, so the same number of waves is spread over all SMs instead: the smallest spc with
// ceil(B / spc) <= waves * SMs (4096 samples: 147 CTAs of 28; a slot left empty costs an idle row of the 8-row DMMA
// tile, nothing else).  `sm_reserve` SMs are left to kernels the caller runs beside this one on other streams.
static int grid2_samples_per_cta(const gpde_vo_plan *pl, int S, long long B, int sm_reserve) {
    if (pl->env.grid2_spc > 0) return std::max(S / 2, std::min(S, pl->env.grid2_spc));
    const long long sms = std::max(1, pl->n_sm - std::max(0, sm_reserve));
    const long long blocks = (B + S - 1) / S, waves = (blocks + sms - 1) / sms;
    const long long spc = (B + waves * sms - 1) / (waves * sms);
    return (int)std::max<long long>((3 * S + 3) / 4, std::min<long long>(S, spc));
}

template <typename TV>
static void grid2_pack(const Grid2Dev &G, const TV *V, int m, int NT, int NX, double *Vp, int n_sm, cudaStream_t st) {
    const long long warps = (long long)(G.ny + 1) * 8;   // one warp per (node row, strip slot)
    const unsigned grid = (unsigned)std::min<long long>((warps + 3) / 4, (long long)n_sm * 16);
    vo_grid2_pack_kernel<TV><<<grid, 128, 0, st>>>(G, V, m, NT, NX, Vp);
}

// TA: conductivities, Dirichlet values and V; TY: y; TR: result (r, or the rho rows of the rho variant)
template <typename TA, typename TY, typename TR>
static int launch_grid2(const gpde_vo_plan *pl, const TA *a, long long a_stride, int a_is_log, const TY *y,
                        const TA *g, long long g_stride, const TA *V, int m, TR *r, void *workspace,
                        int rho_pitch, int sub_f, bool prepacked, long long B, cudaStream_t st, long long y_stride = 0,
                        int sm_reserve = 0) {
    constexpr int EA = (int)sizeof(TA), EY = (int)sizeof(TY);
    if (y_stride == 0) y_stride = pl->dev.d;
    if (y_stride != pl->dev.d && rho_pitch <= 0) return 0;   // only the rho variant is built for strided y
    const bool rho = rho_pitch > 0;
    Grid2Dev G;
    int NT, NX;
    size_t smem;
    if (!grid2_setup(pl, m, rho, sub_f, G, NT, NX, smem, EA, EY)) return 0;
    // y only needs its natural alignment
    if (!grid2_a_aligned(pl, a, a_stride, EA) || ((uintptr_t)y & (EY - 1))) return 0;
    if (!rho && ((uintptr_t)workspace & 15)) return 0;
    const int S = 8 * G.groups;
    double *Vp = (double *)workspace;
    if (!rho && !prepacked) grid2_pack(G, V, m, NT, NX, Vp, pl->n_sm, st);
    unsigned blocks = (unsigned)((B + S - 1) / S);
    // small batches: the node rows of a sample block are cut over the CTAs of a thread-block cluster (SPLIT variant of the
    // kernel) when the blocks alone would leave more than half of the SMs idle; every range gets at least two stages.
    // The cluster size depends on the number of sample blocks only.  GPDE_GRID2_SPLIT=0 keeps one CTA per block.
    int csize = 1;
    if (!rho && std::is_same<TA, TY>::value && std::is_same<TA, TR>::value && pl->env.grid2_split) {
        const int n_stages = G.ny / 2;
        csize = std::min(std::min(8, n_stages / 2), pl->n_sm / (int)blocks);
        if (pl->env.grid2_split > 1) csize = std::min(pl->env.grid2_split, n_stages / 2);   // forced size (tests)
        if (csize < 2 || 2 * (size_t)G.stage_bytes < (size_t)(16 * 8 * 34 + S * 33) * sizeof(double)) csize = 1;
    }
    if (csize == 1) {   // whole samples per CTA: balance the last wave over the SMs
        G.spc = grid2_samples_per_cta(pl, S, B, sm_reserve);
        blocks = (unsigned)((B + G.spc - 1) / G.spc);
    }
    const unsigned grid = blocks * (unsigned)csize;
    // the residual kernel is launched as a programmatic dependent of the packing kernel (its prologue and first
    // a / y stages overlap the packing); with prepacked weights (the packing, if any, was a call of its own) as a
    // dependent of whatever the stream ran before, which it waits for before its first global read: only the launch
    // overlaps
    const bool pdl = !rho && csize == 1;
    G.wait_first = prepacked ? 1 : 0;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(512);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    if (csize > 1) {
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)csize;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
    } else {
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
    }
    cfg.attrs = attr;
    cfg.numAttrs = (pdl || csize > 1) ? 1 : 0;
    const int m_arg = rho ? rho_pitch : m;
    // a_is_log is a template parameter: with the exp() path compiled in or out, each variant gets its own register
    // allocation (as a run-time branch the two paths cost each other 4-8 %, measured A/B)
#define GPDE_LAUNCH_GRID2_YS(NTV, NXV, RHOV, YSV)                                                                \
    {                                                                                                            \
        auto kern = a_is_log ? vo_grid2_kernel<NTV, NXV, RHOV, YSV, true, TA, TY, TR>                           \
                             : vo_grid2_kernel<NTV, NXV, RHOV, YSV, false, TA, TY, TR>;                         \
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));        \
        GPDE_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, G, a, a_stride, a_is_log, y, y_stride, g, g_stride,         \
                                        (const double *)Vp, m_arg, r, B));                                       \
    }
#define GPDE_LAUNCH_GRID2_SPLIT(NTV, NXV)                                                                        \
    {                                                                                                            \
        auto kern = a_is_log ? vo_grid2_kernel<NTV, NXV, false, false, true, TA, TY, TR, true>                   \
                             : vo_grid2_kernel<NTV, NXV, false, false, false, TA, TY, TR, true>;                 \
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));        \
        GPDE_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, G, a, a_stride, a_is_log, y, y_stride, g, g_stride,         \
                                        (const double *)Vp, m_arg, r, B));                                       \
    }
#define GPDE_LAUNCH_GRID2(NTV, NXV, RHOV)                                                                        \
    {                                                                                                            \
        if (csize > 1) { if constexpr (!RHOV && same) GPDE_LAUNCH_GRID2_SPLIT(NTV, NXV) }                        \
        else GPDE_LAUNCH_GRID2_YS(NTV, NXV, RHOV, false)                                                         \
    }
    // instantiated type combinations: (T,T,T) every variant but the strided-y one for FP32; (float,float,double) the rho
    // variant only (rho rows for the FP64 contraction); (T,double,T) the strided-y rho variant only (residual_T)
    constexpr bool same = std::is_same<TA, TY>::value && std::is_same<TA, TR>::value;
    constexpr bool ys_ok = std::is_same<TY, double>::value && std::is_same<TA, TR>::value;
    constexpr bool rho_ok = std::is_same<TA, TY>::value;
    if (rho && y_stride != pl->dev.d) {
        if constexpr (ys_ok) GPDE_LAUNCH_GRID2_YS(1, 0, true, true)
        else return 0;
    } else if (rho) {
        if constexpr (rho_ok) GPDE_LAUNCH_GRID2(1, 0, true)
        else return 0;
    } else if constexpr (same) {
        if (NT == 1 && NX == 0) GPDE_LAUNCH_GRID2(1, 0, false)
        else if (NT == 1) GPDE_LAUNCH_GRID2(1, 1, false)
        else if (NT == 2 && NX == 0) GPDE_LAUNCH_GRID2(2, 0, false)
        else if (NT == 2) GPDE_LAUNCH_GRID2(2, 1, false)
        else if (NT == 3 && NX == 0) GPDE_LAUNCH_GRID2(3, 0, false)
        else if (NT == 3) GPDE_LAUNCH_GRID2(3, 1, false)
        else GPDE_LAUNCH_GRID2(4, 0, false)
    } else {
        return 0;
    }
#undef GPDE_LAUNCH_GRID2
#undef GPDE_LAUNCH_GRID2_SPLIT
#undef GPDE_LAUNCH_GRID2_YS
    GPDE_CUDA_OK(cudaGetLastError());
    return 1;
}

// Transposed application q = K_ff(a) (V s) on the reference's pixel meshes in ONE kernel (WT variant of vo_grid2_kernel):
// V^T packed in fragment order (vo_grid2_pack_t_kernel, 4 us), then the marching kernel produces the rows of w = s V^T
// in shared memory itself.  Returns 1 if it served the call, 0 if the two-kernel route should (mesh / alignment / shared
// memory), <0 on error.  s, V and a share the element type T; q too.
template <typename T>
static int launch_grid2_wt(const gpde_vo_plan *pl, const T *a, long long a_stride, int a_is_log, const T *V, int mw, const T *s,
                           T *q, void *workspace, long long B, cudaStream_t st) {
    constexpr int EA = (int)sizeof(T);
    if (!pl->env.fused_t || mw < 1 || mw > 32) return 0;
    Grid2Dev G;
    int NT, NX;
    size_t smem;
    if (!grid2_setup(pl, 0, true, 0, G, NT, NX, smem, EA, 8)) return 0;
    if (!grid2_a_aligned(pl, a, a_stride, EA) || ((uintptr_t)workspace & 15)) return 0;
    const int KS = mw <= 16 ? 4 : (mw <= 28 ? 7 : 8);
    G.v_row_bytes = G.nstrips * 2 * KS * 256 + kGrid2MaskBytes;
    const size_t fixed = smem;                  // (rho variant: no V stages counted yet)
    G.nvs = (fixed + 3 * 2 * (size_t)G.v_row_bytes <= 227 * 1024) ? 3 : 2;
    smem = fixed + (size_t)G.nvs * 2 * G.v_row_bytes;
    if (smem > 227 * 1024) return 0;
    const int S = 8 * G.groups, d = pl->dev.d;
    double *Vp = (double *)workspace;
    {
        const long long warps = (long long)(G.ny + 1) * 8;   // one warp per (node row, strip slot)
        const unsigned grid = (unsigned)std::min<long long>((warps + 3) / 4, (long long)pl->n_sm * 16);
        vo_grid2_pack_t_kernel<T><<<grid, 128, 0, st>>>(G, V, mw, KS, Vp);
    }
    G.spc = grid2_samples_per_cta(pl, S, B, 0);
    const unsigned blocks = (unsigned)((B + G.spc - 1) / G.spc);
#define GPDE_LAUNCH_GRID2_WT(KSV)                                                                                \
    {                                                                                                            \
        auto kern = a_is_log ? vo_grid2_kernel<1, 0, true, false, true, T, double, T, false, KSV>                \
                             : vo_grid2_kernel<1, 0, true, false, false, T, double, T, false, KSV>;              \
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));        \
        kern<<<blocks, 512, smem, st>>>(G, a, a_stride, a_is_log, (const double *)nullptr, 0ll, s, (long long)mw, \
                                        (const double *)Vp, d, q, B);                                            \
    }
    if (KS == 4) GPDE_LAUNCH_GRID2_WT(4)
    else if (KS == 7) GPDE_LAUNCH_GRID2_WT(7)
    else GPDE_LAUNCH_GRID2_WT(8)
#undef GPDE_LAUNCH_GRID2_WT
    GPDE_CUDA_OK(cudaGetLastError());
    return 1;
}

// Structured-grid path.  Returns 1 if it served the call, 0 if the caller should use the generic kernels (alignment /
// size conditions not met), <0 on error.
template <typename T>
static int launch_grid_lean(const gpde_vo_plan *pl, const T *a, long long a_stride, int a_is_log, const T *y,
                            const T *g, long long g_stride, const T *V, int m, T *r, void *workspace,
                            int sub_f, bool prepacked, long long B, cudaStream_t st, int sm_reserve = 0) {
    if (!y || m < 1 || m > 32) return 0;
    const int rc2 = launch_grid2<T, T, T>(pl, a, a_stride, a_is_log, y, g, g_stride, V, m, r, workspace, 0, sub_f, prepacked, B, st, 0,
                                          sm_reserve);
    if (rc2 != 0) return rc2;
    if (prepacked)
        return fail(GPDE_ERR_ARG, "vo_residual: packed weights (flags bit1) need the lean structured-grid kernel for this call "
                                  "(16-byte aligned a and sample stride, y given, no load vector)");
    return 0;
}

// Structured-grid fine residual rho[B][pitch] (pitch >= d, padding zeroed) for the tensor-core contraction.
// Returns 1 if it served the call, 0 if the generic matvec kernel should (alignment / size), <0 on error.
template <typename T, typename TR>
static int launch_grid_rho_lean(const gpde_vo_plan *pl, const T *a, long long a_stride, int a_is_log, const T *y,
                                const T *g, long long g_stride, TR *rho, int pitch, int sub_f, long long B, cudaStream_t st) {
    if (!y) return 0;
    return launch_grid2<T, T, TR>(pl, a, a_stride, a_is_log, y, g, g_stride, (const T *)nullptr, 0, rho, nullptr, pitch, sub_f,
                                  false, B, st);
}
template <typename Ta, typename Ty, typename To>
static int launch_matvec(const gpde_vo_plan *pl, const Ta *a, long long a_stride, int a_is_log, const Ty *y,
                         const Ta *g, long long g_stride, int sub_f, double *rho_ws, int ws_stride, To *rho_out,
                         long long B, cudaStream_t st) {
    const VoDev &P = pl->dev;
    const size_t per = sizeof(double) * (size_t)P.n_inputs;
    const size_t cap = 200 * 1024;
    const int nsm = pl->n_sm;
    int S = 1;
    if (B >= 4LL * nsm * 2 && 4 * per <= cap) S = 4;
    else if (B >= 2LL * nsm * 2 && 2 * per <= cap) S = 2;
    const int stage = (S * per <= cap) ? 1 : 0;
    const size_t smem = stage ? S * per : 0;
    const long long ctas = (B + S - 1) / S;
    const unsigned grid = (unsigned)std::min<long long>(ctas, (long long)nsm * 8);
#define GPDE_LAUNCH_MV(SS)                                                                               \
    {                                                                                                    \
        auto kern = vo_matvec_kernel<Ta, Ty, To, SS>;                                                    \
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        kern<<<grid, kVoThreads, smem, st>>>(P, a, a_stride, a_is_log, y, g, g_stride, sub_f, rho_ws,    \
                                             ws_stride, rho_out, B, stage);                               \
    }
    if (S == 4) GPDE_LAUNCH_MV(4)
    else if (S == 2) GPDE_LAUNCH_MV(2)
    else GPDE_LAUNCH_MV(1)
#undef GPDE_LAUNCH_MV
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

// Many weighting functions on the reference's pixel meshes: rho produced inside the contraction kernel (vo_gridgemm.cuh).
// Returns 1 if it served the call, 0 if the two-kernel route should, < 0 on error.
static bool gridgemm_setup(const gpde_vo_plan *pl, int m, int sub_f, int elem, GGDev &G, int &bn, int &nw, size_t &smem) {
    Grid2Dev G2;
    int nt2, nx2;
    size_t smem2;
    if (!pl->env.gridgemm || m <= 32 || !use_grid(pl) || !grid2_setup(pl, 0, true, sub_f, G2, nt2, nx2, smem2, elem, elem)) return false;
    memset(&G, 0, sizeof(G));
    G.nx = G2.nx; G.ny = G2.ny; G.ncol = G2.ncol; G.nstrips = G2.nstrips;
    G.in0 = G2.in0; G.sy = G2.sy; G.rh = G2.rh; G.scale = G2.scale;
    bn = m <= 128 ? 128 : 256;
    G.ctiles = (m + bn - 1) / bn;
    nw = 8;   // node columns per producer warp: 4 producer warps (8 warps of 4 columns measured slower: 4.46 vs 4.26 ms at config 3)
    for (G.stages_b = 4; G.stages_b >= 3; --G.stages_b)
        if ((smem = gg_smem_bytes(bn, G.stages_b, elem, nw)) <= 227 * 1024) return true;
    return false;
}
static size_t gridgemm_workspace_bytes(const gpde_vo_plan *pl, long long B, int m) {
    GGDev G;
    int bn, nw;
    size_t smem;
    if (!gridgemm_setup(pl, m, 0, 8, G, bn, nw, smem)) return 0;
    // packed V | partial tiles of the split contraction | conductivities of a log-field input
    return gg_packed_bytes(bn, G.ctiles, G.nstrips * (G.ny + 1)) + 32 + sizeof(double) * 8 * (size_t)B * G.ctiles * bn +
           sizeof(double) * (size_t)B * pl->dev.n_inputs;
}
template <typename T>
static int launch_gridgemm(const gpde_vo_plan *pl, const T *a, long long a_stride, int a_is_log, const T *y, const T *g,
                           long long g_stride, const T *V, int m, T *r, void *workspace, int sub_f, long long B,
                           cudaStream_t st) {
    GGDev G;
    int bn, nw;
    size_t smem;
    if (((uintptr_t)workspace & 15) || !gridgemm_setup(pl, m, sub_f, (int)sizeof(T), G, bn, nw, smem)) return 0;
    // the producers address a warp's 32 samples by 32-bit byte offsets
    const long long span = 32 * std::max<long long>(std::max<long long>(pl->dev.d, a_stride), g_stride) + 2 * (long long)pl->dev.d;
    if (span * (long long)sizeof(T) >= (1ll << 31)) return 0;
    const int chunks = G.nstrips * (G.ny + 1);
    double *Vp = (double *)workspace;
    const long long tiles = (B + kGGBM - 1) / kGGBM * G.ctiles;
    int splits = pl->env.gemm_splits > 0 ? pl->env.gemm_splits : gemm_splits(tiles, pl->n_sm, chunks);
    splits = std::max(1, std::min(splits, G.nstrips));
    const int ldp = G.ctiles * bn;
    double *part0 = (double *)(((uintptr_t)Vp + gg_packed_bytes(bn, G.ctiles, chunks) + 15) & ~(uintptr_t)15);
    double *partial = splits > 1 ? part0 : nullptr;
    if (a_is_log) {   // conductivities by one streaming pass (behind the partial tiles in the workspace)
        T *cond = (T *)(((uintptr_t)(part0 + (size_t)8 * B * ldp) + 15) & ~(uintptr_t)15);
        const long long n = a_stride ? B * a_stride : (long long)pl->dev.n_inputs;
        if (a_stride && a_stride != pl->dev.n_inputs) return 0;
        vo_exp_rows_kernel<T><<<(unsigned)std::min<long long>((n + 255) / 256, (long long)pl->n_sm * 16), 256, 0, st>>>(a, n, cond);
        a = cond;
    }
    const dim3 grid((unsigned)((B + kGGBM - 1) / kGGBM), (unsigned)G.ctiles, (unsigned)splits);
    const unsigned pgrid = (unsigned)std::min<long long>(((long long)G.ctiles * chunks + 7) / 8, (long long)pl->n_sm * 8);
#define GPDE_LAUNCH_GG(BNV, NWV)                                                                                  \
    {                                                                                                             \
        vo_gridgemm_pack_kernel<BNV, T><<<pgrid, 256, 0, st>>>(G, V, m, Vp);                                      \
        auto kern = vo_gridgemm_kernel<BNV, NWV, T, T>;                                                           \
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));         \
        kern<<<grid, gg_threads(NWV), smem, st>>>(G, a, a_stride, y, g, g_stride, Vp, r, m, ldp, B, partial);     \
    }
    if (bn == 128) GPDE_LAUNCH_GG(128, 8) else GPDE_LAUNCH_GG(256, 8)
#undef GPDE_LAUNCH_GG
    GPDE_CUDA_OK(cudaGetLastError());
    if (splits > 1) {
        const long long total = B * m;
        const unsigned rgrid = (unsigned)std::min<long long>((total + 255) / 256, (long long)pl->n_sm * 16);
        vo_gemm_reduce_kernel<T><<<rgrid, 256, 0, st>>>(partial, splits, ldp, r, m, B);
        GPDE_CUDA_OK(cudaGetLastError());
    }
    return 1;
}

template <typename T>
static int vo_residual(const gpde_vo_plan *pl, const T *a, int64_t a_stride, int a_is_log, const T *y, const T *g,
                       int64_t g_stride, const T *V, int64_t v_stride, int m, T *r, T *rho, void *workspace, int flags,
                       int64_t B, gpde_stream_t stream) {
    if (!pl || B < 0 || m < 0) return fail(GPDE_ERR_ARG, "vo_residual: bad argument");
    if (v_stride != 0 && (m == 0 || v_stride != (int64_t)pl->dev.d * m))
        return fail(GPDE_ERR_ARG, "vo_residual: v_stride must be 0, or d*m with m > 0");
    if (B == 0) return GPDE_OK;
    if (!a) return fail(GPDE_ERR_ARG, "vo_residual: null conductivity field");
    if (m > 0 && (!V || !r)) return fail(GPDE_ERR_ARG, "vo_residual: V and r are required when m > 0");
    if (m > 0 && !workspace) return fail(GPDE_ERR_ARG, "vo_residual: workspace required");
    if (m == 0 && !rho) return fail(GPDE_ERR_ARG, "vo_residual: nothing to compute");
    if (v_stride) {   // r_b = V_b^T rho_b: the rho-only residual (whichever kernel the plan picks for it), then the contraction
        if ((uintptr_t)workspace & 15) return fail(GPDE_ERR_ARG, "vo_residual: a per-sample V needs a 16-byte aligned workspace");
        if (flags & 2) return fail(GPDE_ERR_ARG, "vo_residual: packed weights (flags bit1) are a shared-V layout");
        T *rb = rho ? rho : (T *)workspace;   // rho [B,d]: the caller's, else the workspace
        const int rc = vo_residual<T>(pl, a, a_stride, a_is_log, y, g, g_stride, nullptr, 0, 0, nullptr, rb, nullptr, flags & 1,
                                      B, stream);
        if (rc != GPDE_OK) return rc;
        DeviceGuard guard(pl->device);
        const int npan = (m + kVbPanel - 1) / kVbPanel;
        const unsigned grid = (unsigned)std::min<long long>((long long)B * npan, (long long)pl->n_sm * 64);
        vo_vb_contract_kernel<T><<<grid, kVbThreads, 0, (cudaStream_t)stream>>>(V, rb, r, pl->dev.d, m, (long long)B);
        GPDE_CUDA_OK(cudaGetLastError());
        return GPDE_OK;
    }
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (m > 0 && !rho && use_grid(pl)) {
        const int rc = launch_grid_lean<T>(pl, a, (long long)a_stride, a_is_log, y, g, (long long)g_stride, V, m, r, workspace,
                                           (flags & 1) ? 0 : 1, (flags & 2) != 0, (long long)B, st, (flags >> 8) & 0xff);
        if (rc != 0) return rc < 0 ? rc : GPDE_OK;
    }
    if (m == 0 && rho && use_grid(pl)) {   // the fine residual alone: rho rows straight into the caller's [B,d]
        const int rc = launch_grid_rho_lean<T, T>(pl, a, (long long)a_stride, a_is_log, y, g, (long long)g_stride, rho, pl->dev.d,
                                                  (flags & 1) ? 0 : 1, (long long)B, st);
        if (rc != 0) return rc < 0 ? rc : GPDE_OK;
    }
    if (flags & 2) return fail(GPDE_ERR_ARG, "vo_residual: packed weights (flags bit1) are not usable for this call");
    if (m > 0 && m <= 32 && use_fused(pl)) {
        const unsigned grid = (unsigned)((B + kFS - 1) / kFS);
        const int sub_f = (flags & 1) ? 0 : 1;
        constexpr bool kCanAsync = sizeof(T) == 8;
        const bool use_async = kCanAsync && pl->tiles.async_ok && !pl->env.sync_staging;
#define GPDE_LAUNCH_FUSED(WN)                                                                                  \
    {                                                                                                          \
        auto kern = use_async ? vo_fused_kernel<T, WN, kCanAsync> : vo_fused_kernel<T, WN, false>;             \
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl->fused_smem)); \
        kern<<<grid, kFT, pl->fused_smem, st>>>(pl->dev, pl->tiles, a, (long long)a_stride, a_is_log, y, g,   \
                                                (long long)g_stride, V, m, r, rho, sub_f, (long long)B);       \
    }
        if (m <= 8) GPDE_LAUNCH_FUSED(1)
        else if (m <= 16) GPDE_LAUNCH_FUSED(2)
        else GPDE_LAUNCH_FUSED(4)
#undef GPDE_LAUNCH_FUSED
        GPDE_CUDA_OK(cudaGetLastError());
        return GPDE_OK;
    }
    if (m > 32 && !rho && use_grid(pl)) {   // many weighting functions on a pixel mesh: one kernel, rho never leaves the SM
        const int rc = launch_gridgemm<T>(pl, a, (long long)a_stride, a_is_log, y, g, (long long)g_stride, V, m, r, workspace,
                                          (flags & 1) ? 0 : 1, (long long)B, st);
        if (rc != 0) return rc < 0 ? rc : GPDE_OK;
    }
    // version 1: rho -> K-padded workspace, then the FP64 tensor-core contraction (vo_gemm.cuh)
    const int d = pl->dev.d, dp = gemm_dp(d);
    double *ws = m > 0 ? (double *)workspace : nullptr;
    int rc = 0;
    if (m > 0 && !rho && use_grid(pl)) {   // structured pixel grid: the marching kernel produces rho (no V inside)
        rc = launch_grid_rho_lean<T, double>(pl, a, (long long)a_stride, a_is_log, y, g, (long long)g_stride, ws, dp,
                                             (flags & 1) ? 0 : 1, (long long)B, st);
        if (rc < 0) return rc;
    }
    if (rc == 0) {
        rc = launch_matvec<T, T, T>(pl, a, a_stride, a_is_log, y, g, g_stride, (flags & 1) ? 0 : 1, ws, dp, rho, B, st);
        if (rc != GPDE_OK) return rc;
    }
    if (m > 0) {
        const int bn = gemm_bn(m), ldb = gemm_ldb(m);
        double *Vp = ws + (size_t)B * dp;
        {
            const long long total = (long long)dp * ldb;
            const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, (long long)pl->n_sm * 8);
            vo_gemm_pack_kernel_t<T><<<grid, 256, 0, st>>>(V, d, m, Vp, dp, ldb);
        }
        dim3 grid((unsigned)((B + kGemmBM - 1) / kGemmBM), (unsigned)(ldb / bn));
        // tail of the tile grid on the SMs: parts of the contraction length with a deterministic reduction (vo_gemm.cuh)
        const int splits = pl->env.gemm_splits > 0 ? pl->env.gemm_splits
                                                   : gemm_splits((long long)grid.x * grid.y, pl->n_sm, dp / kGemmKC);
        double *partial = splits > 1 ? Vp + (size_t)dp * ldb : nullptr;
        grid.z = (unsigned)splits;
        const size_t smem = gemm_smem(bn);
        if (bn == 64) {
            auto kern = vo_gemm_kernel<64, T>;
            GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<grid, kGemmThreads, smem, st>>>(ws, dp, Vp, ldb, r, m, (long long)B, partial);
        } else {
            auto kern = vo_gemm_kernel<128, T>;
            GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<grid, kGemmThreads, smem, st>>>(ws, dp, Vp, ldb, r, m, (long long)B, partial);
        }
        GPDE_CUDA_OK(cudaGetLastError());
        if (splits > 1) {
            const long long total = (long long)B * m;
            const unsigned rgrid = (unsigned)std::min<long long>((total + 255) / 256, (long long)pl->n_sm * 16);
            vo_gemm_reduce_kernel<T><<<rgrid, 256, 0, st>>>(partial, splits, ldb, r, m, (long long)B);
            GPDE_CUDA_OK(cudaGetLastError());
        }
    }
    return GPDE_OK;
}

// w = s V^T [B, ldw] in FP64 into `workspace` (16-byte aligned, >= expand_bytes): the first half of residual_T's two-kernel
// route on pixel grids and of the residual gradient (vo_grad.cuh).  FP32 I/O: s and V converted on load.
static size_t expand_bytes(const gpde_vo_plan *pl, long long B, int m) {
    const size_t d = (size_t)pl->dev.d;
    if (m <= 32) return sizeof(double) * (size_t)B * ((d + 3) & ~(size_t)3);
    const size_t mp = (size_t)gemm_dp(m), ldb = (d + 127) / 128 * 128;
    return sizeof(double) * ((size_t)B * mp + mp * ldb + (size_t)B * d);
}
template <typename T>
static int launch_expand(const gpde_vo_plan *pl, const T *s, const T *V, int m, void *workspace, long long B, cudaStream_t st,
                         double *&w, long long &ldw) {
    const int d = pl->dev.d;
    w = (double *)workspace;
    ldw = d;
    if (m <= 32) {   // contraction length m <= 32: one launch, operands read in place (vo_expand.cuh)
        ldw = ((long long)d + 3) & ~3ll;
        const int n_tiles = (d + 7) / 8;
        const unsigned gx = (unsigned)((B + 8 * kExpandMT * kExpandWarps - 1) / (8 * kExpandMT * kExpandWarps));
        const int nch = std::max(1, std::min(n_tiles, (int)(4 * pl->n_sm / gx)));
        const int tpc = std::min((n_tiles + nch - 1) / nch, 64);         // <= 64 n-tiles of V per CTA in shared memory
        const dim3 grid(gx, (unsigned)((n_tiles + tpc - 1) / tpc));
        const size_t smem = (size_t)tpc * 8 * kExpandVPitch * sizeof(double);
#define GPDE_LAUNCH_EXPAND(KSV)                                                                                     \
    {                                                                                                           \
        auto kern = vo_expand_dmma_kernel<KSV, T>;                                                              \
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));       \
        kern<<<grid, kExpandWarps * 32, smem, st>>>(s, V, w, ldw, (long long)B, d, m, tpc);                     \
    }
        if (m <= 8) GPDE_LAUNCH_EXPAND(2)
        else if (m <= 16) GPDE_LAUNCH_EXPAND(4)
        else if (m <= 28) GPDE_LAUNCH_EXPAND(7)
        else GPDE_LAUNCH_EXPAND(8)
#undef GPDE_LAUNCH_EXPAND
        GPDE_CUDA_OK(cudaGetLastError());
    } else if constexpr (sizeof(T) == 8) {   // m > 32: the general FP64 GEMM, w [B,d] behind the padded operands
        const int mp = gemm_dp(m), bn = 128, ldb = (d + bn - 1) / bn * bn;
        double *Sp = (double *)workspace, *Vt = Sp + (size_t)B * mp;
        w = Vt + (size_t)mp * ldb;
        {
            const long long total = (long long)B * mp;
            const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, (long long)pl->n_sm * 8);
            vo_gemm_pad_rows_kernel<<<grid, 256, 0, st>>>(s, (long long)B, m, Sp, mp);
            vo_gemm_pack_transposed_kernel<<<dim3((unsigned)(ldb / 32), (unsigned)((mp + 31) / 32)), dim3(32, 8), 0, st>>>(
                V, d, m, Vt, mp, ldb);
        }
        {
            auto kern = vo_gemm_kernel<128, double>;
            const size_t smem = gemm_smem(bn);
            GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            dim3 grid((unsigned)((B + kGemmBM - 1) / kGemmBM), (unsigned)(ldb / bn));
            kern<<<grid, kGemmThreads, smem, st>>>(Sp, mp, Vt, ldb, w, d, (long long)B, (double *)nullptr);
            GPDE_CUDA_OK(cudaGetLastError());
        }
    } else {   // m > 32 with FP32 I/O
        const long long total = B * (long long)d;
        const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, (long long)pl->n_sm * 16);
        vo_expand_kernel<T><<<grid, 256, 0, st>>>(s, V, w, B, d, m);
        GPDE_CUDA_OK(cudaGetLastError());
    }
    return GPDE_OK;
}

// One weighting matrix per sample (vo_vb.cuh): w_b = V_b s_b, FP64 rows of pitch ldw.  The rows are padded to 4 doubles
// (vb_ldw) for the strided-y marching kernel, as launch_expand pads them.
static long long vb_ldw(const gpde_vo_plan *pl) { return ((long long)pl->dev.d + 3) & ~3ll; }
template <typename T>
static int launch_vb_expand(const gpde_vo_plan *pl, const T *V, const T *s, int m, double *w, long long ldw, long long B,
                            cudaStream_t st) {
    const long long jobs = B * ((pl->dev.d + kVbRows - 1) / kVbRows);
    const unsigned grid = (unsigned)std::min<long long>(jobs, (long long)pl->n_sm * 64);
    vo_vb_expand_kernel<T><<<grid, kVbExpThreads, 0, st>>>(V, s, w, ldw, pl->dev.d, m, B);
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

template <typename T>
static int vo_residual_T(const gpde_vo_plan *pl, const T *a, int64_t a_stride, int a_is_log, const T *V, int64_t v_stride,
                         int m, const T *s, T *q, void *workspace, int64_t B, gpde_stream_t stream) {
    if (!pl || m <= 0 || B < 0) return fail(GPDE_ERR_ARG, "vo_residual_T: bad argument");
    if (v_stride != 0 && v_stride != (int64_t)pl->dev.d * m) return fail(GPDE_ERR_ARG, "vo_residual_T: v_stride must be 0 or d*m");
    if (B == 0) return GPDE_OK;
    if (!a || !V || !s || !q || !workspace) return fail(GPDE_ERR_ARG, "vo_residual_T: null argument");
    if (v_stride && ((uintptr_t)workspace & 15))
        return fail(GPDE_ERR_ARG, "vo_residual_T: a per-sample V needs a 16-byte aligned workspace");
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (!v_stride && use_grid(pl) && m <= 32) {   // one kernel: w = s V^T never leaves the SM
        const int rc = launch_grid2_wt<T>(pl, a, (long long)a_stride, a_is_log, V, m, s, q, workspace, (long long)B, st);
        if (rc != 0) return rc < 0 ? rc : GPDE_OK;
    }
    // structured pixel grid: w = s V^T on the FP64 tensor pipe (per-sample V: the expansion kernel), then q = K_ff w with the
    // marching kernel (rho of u~ = (w, 0) without the load vector IS K_ff w); FP32 I/O: s and V converted on load, w stays
    // FP64, a staged and q stored as floats
    Grid2Dev G2;
    int nt2, nx2;
    size_t smem2;
    const bool on_grid = use_grid(pl) && (v_stride || m <= 32 || sizeof(T) == 8) &&
                         grid2_a_aligned(pl, a, (long long)a_stride, (int)sizeof(T)) && !((uintptr_t)workspace & 15) &&
                         grid2_setup(pl, 0, true, 0, G2, nt2, nx2, smem2, (int)sizeof(T), 8);
    if (!on_grid && !v_stride && use_fused(pl) && sizeof(double) * kFS * (size_t)m <= sizeof(double) * kFS * kRhoPitch) {
        const unsigned grid = (unsigned)((B + kFS - 1) / kFS);
        const size_t smem = pl->fused_smem;   // the coefficient vectors live in the (unused) rho tile
        auto kern = vo_fused_T_kernel<T>;
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, kFT, smem, st>>>(pl->dev, pl->tiles, a, (long long)a_stride, a_is_log, V, m, s, q, (long long)B);
        GPDE_CUDA_OK(cudaGetLastError());
        return GPDE_OK;
    }
    const int d = pl->dev.d;
    double *w = (double *)workspace;
    long long ldw = d;   // the generic matvec reads w with pitch d
    if (v_stride) {
        if (on_grid) ldw = vb_ldw(pl);
        const int rce = launch_vb_expand<T>(pl, V, s, m, w, ldw, (long long)B, st);
        if (rce != GPDE_OK) return rce;
    } else if (on_grid) {
        const int rce = launch_expand<T>(pl, s, V, m, workspace, (long long)B, st, w, ldw);
        if (rce != GPDE_OK) return rce;
    } else {
        const long long total = B * (long long)d;
        const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, (long long)pl->n_sm * 16);
        vo_expand_kernel<T><<<grid, 256, 0, st>>>(s, V, w, B, d, m);
        GPDE_CUDA_OK(cudaGetLastError());
    }
    if (on_grid) {
        const int rc = launch_grid2<T, double, T>(pl, a, (long long)a_stride, a_is_log, w, nullptr, 0, nullptr, 0, q, nullptr, d, 0,
                                                  false, (long long)B, st, ldw);
        if (rc != 0) return rc < 0 ? rc : GPDE_OK;
        return fail(GPDE_ERR_ARG, "vo_residual_T: lean grid kernel declined after setup");
    }
    return launch_matvec<T, double, T>(pl, a, a_stride, a_is_log, w, (const T *)nullptr, 0, 0, (double *)nullptr, 0, q, B, st);
}

// grad_a (marching kernel on pixel grids, per-input cell lists otherwise) and grad_g (Dirichlet rows of K(a)) from
// w = the rows V gbar_r_b (FP64, pitch ldw).  The kernel choice depends on the plan only.
template <typename T>
static int launch_grad(const gpde_vo_plan *pl, const T *a, int64_t a_stride, int a_is_log, const T *y, const T *g,
                       int64_t g_stride, const double *w, long long ldw, T *grad_a, T *grad_g, int64_t B, cudaStream_t st) {
    const int d = pl->dev.d;
    if (grad_a && pl->grid.ok) {
        const GridDev &G = pl->grid;
        const long long total = (long long)B * G.nx;
        const unsigned grid = (unsigned)std::min<long long>((total + kGradThreads - 1) / kGradThreads, (long long)pl->n_sm * 8);
        vo_grad_grid_kernel<T><<<grid, kGradThreads, 0, st>>>(G.nx, G.ny, G.in0, G.sy, -G.rh * G.scale, -G.scale, a,
                                                                (long long)a_stride, a_is_log, y, d, g, (long long)g_stride,
                                                                w, ldw, grad_a, (long long)B);
        GPDE_CUDA_OK(cudaGetLastError());
    } else if (grad_a) {
        const long long total = (long long)B * pl->dev.n_inputs;
        const unsigned grid = (unsigned)std::min<long long>((total + kGradThreads - 1) / kGradThreads, (long long)pl->n_sm * 16);
        vo_grad_cells_kernel<T><<<grid, kGradThreads, 0, st>>>(pl->grad, a, (long long)a_stride, a_is_log, y, d, g,
                                                                 (long long)g_stride, w, ldw, grad_a, (long long)B);
        GPDE_CUDA_OK(cudaGetLastError());
    }
    if (grad_g && pl->dev.n_bc > 0) {
        const long long total = (long long)B * pl->dev.n_bc;
        const unsigned grid = (unsigned)std::min<long long>((total + kGradThreads - 1) / kGradThreads, (long long)pl->n_sm * 16);
        vo_grad_g_kernel<T><<<grid, kGradThreads, 0, st>>>(pl->grad.bc_rows, a, (long long)a_stride, a_is_log, w, ldw, grad_g,
                                                             (long long)B);
        GPDE_CUDA_OK(cudaGetLastError());
    }
    return GPDE_OK;
}

// gpde_vo_residual_grad_*: w = gbar_r V^T (per-sample V: w_b = V_b gbar_r_b), then launch_grad.
template <typename T>
static int vo_residual_grad(const gpde_vo_plan *pl, const T *a, int64_t a_stride, int a_is_log, const T *y, const T *g,
                            int64_t g_stride, const T *V, int64_t v_stride, int m, const T *gbar_r, T *grad_a, T *grad_g,
                            void *workspace, int64_t B, gpde_stream_t stream) {
    if (!pl || B < 0) return fail(GPDE_ERR_ARG, "vo_residual_grad: bad argument (null plan or B < 0)");
    if (m <= 0) return fail(GPDE_ERR_ARG, "vo_residual_grad: m = %d weighting functions (must be > 0)", m);
    if (a_stride != 0 && a_stride != pl->dev.n_inputs)
        return fail(GPDE_ERR_ARG, "vo_residual_grad: a_stride must be 0 or n_inputs = %d", pl->dev.n_inputs);
    if (g_stride != 0 && g_stride != pl->dev.n_bc)
        return fail(GPDE_ERR_ARG, "vo_residual_grad: g_stride must be 0 or n_bc = %d", pl->dev.n_bc);
    if (v_stride != 0 && v_stride != (int64_t)pl->dev.d * m)
        return fail(GPDE_ERR_ARG, "vo_residual_grad: v_stride must be 0 or d*m");
    if (B == 0) return GPDE_OK;
    if (!V || !gbar_r) return fail(GPDE_ERR_ARG, "vo_residual_grad: V and gbar_r are required");
    if (!a) return fail(GPDE_ERR_ARG, "vo_residual_grad: null conductivity field");
    if (!workspace || ((uintptr_t)workspace & 15))
        return fail(GPDE_ERR_ARG, "vo_residual_grad: workspace must be non-NULL and 16-byte aligned "
                                  "(>= gpde_vo_workspace_bytes)");
    if (!grad_a && !grad_g) return GPDE_OK;
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    double *w = (double *)workspace;
    long long ldw = vb_ldw(pl);
    const int rce = v_stride ? launch_vb_expand<T>(pl, V, gbar_r, m, w, ldw, (long long)B, st)
                             : launch_expand<T>(pl, gbar_r, V, m, workspace, (long long)B, st, w, ldw);
    if (rce != GPDE_OK) return rce;
    return launch_grad<T>(pl, a, a_stride, a_is_log, y, g, g_stride, w, ldw, grad_a, grad_g, B, st);
}

// gpde_vo_energy_step_f64 for MP = 32 or 64 (vo_energy.cuh)
template <int MP>
int vo_energy_step_launch(const gpde_vo_plan *pl, const double *a, int64_t a_stride, const double *V, int64_t v_stride,
                          int m, const double *rho, const double *g, const double *prec, const double *inv_T,
                          double *mean, int *info, int64_t N, cudaStream_t st) {
    auto kern = vo_energy_step_kernel<MP>;
    const size_t smem = energy_smem_bytes<MP>(pl->csr.max_row);
    GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)N, kPostThreads, smem, st>>>(pl->csr, a, (long long)a_stride, V, (long long)v_stride, m, rho, g, prec,
                                                  inv_T, mean, info);
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

}  // namespace gpde

using namespace gpde;

extern "C" {

int gpde_vo_plan_create(gpde_vo_plan **plan, int n_nodes, int n_cells, const int32_t *cell_dofs, const double *Ke,
                        const int32_t *cell_to_input, int n_inputs, const int64_t *free_dofs, int d,
                        const int64_t *bc_dofs, int n_bc, const double *f_full, int device) {
    if (!plan || !cell_dofs || !Ke || !cell_to_input || !free_dofs || n_nodes <= 0 || n_cells <= 0 ||
        n_inputs <= 0 || d <= 0 || n_bc < 0 || (n_bc > 0 && !bc_dofs))
        return fail(GPDE_ERR_ARG, "vo_plan_create: bad argument");
    std::vector<int> src(n_nodes, INT32_MIN);   // node -> encoded source
    for (int i = 0; i < d; ++i) {
        if (free_dofs[i] < 0 || free_dofs[i] >= n_nodes) return fail(GPDE_ERR_ARG, "vo_plan_create: free dof range");
        src[free_dofs[i]] = i;
    }
    for (int c = 0; c < n_bc; ++c) {
        if (bc_dofs[c] < 0 || bc_dofs[c] >= n_nodes) return fail(GPDE_ERR_ARG, "vo_plan_create: bc dof range");
        if (src[bc_dofs[c]] != INT32_MIN) return fail(GPDE_ERR_ARG, "vo_plan_create: dof both free and constrained");
        src[bc_dofs[c]] = -c - 1;
    }
    for (int v = 0; v < n_nodes; ++v)
        if (src[v] == INT32_MIN) return fail(GPDE_ERR_ARG, "vo_plan_create: node %d neither free nor constrained", v);
    // incident cells per free row
    std::vector<int> count(d, 0);
    for (int c = 0; c < n_cells; ++c) {
        if (cell_to_input[c] < 0 || cell_to_input[c] >= n_inputs)
            return fail(GPDE_ERR_ARG, "vo_plan_create: cell_to_input out of range");
        for (int l = 0; l < 3; ++l) {
            const int v = cell_dofs[3 * c + l];
            if (v < 0 || v >= n_nodes) return fail(GPDE_ERR_ARG, "vo_plan_create: cell dof out of range");
            if (src[v] >= 0) count[src[v]]++;
        }
    }
    int nslots = 0;
    for (int i = 0; i < d; ++i) nslots = std::max(nslots, count[i]);
    const size_t tot = (size_t)nslots * d;
    std::vector<int> ell_in(tot, 0), ell_j1(tot), ell_j2(tot);
    std::vector<double> c0(tot, 0.0), c1(tot, 0.0), c2(tot, 0.0);
    for (size_t k = 0; k < tot; ++k) ell_j1[k] = ell_j2[k] = (int)(k % d);   // padding: self, zero coefficients
    std::fill(count.begin(), count.end(), 0);
    for (int c = 0; c < n_cells; ++c)
        for (int l = 0; l < 3; ++l) {
            const int v = cell_dofs[3 * c + l];
            if (src[v] < 0) continue;
            const int i = src[v], t = count[i]++;
            const int l1 = (l + 1) % 3, l2 = (l + 2) % 3;
            const size_t k = (size_t)t * d + i;
            ell_in[k] = cell_to_input[c];
            ell_j1[k] = src[cell_dofs[3 * c + l1]];
            ell_j2[k] = src[cell_dofs[3 * c + l2]];
            c0[k] = Ke[9 * c + 3 * l + l];
            c1[k] = Ke[9 * c + 3 * l + l1];
            c2[k] = Ke[9 * c + 3 * l + l2];
        }
    std::vector<double> f_free(d, 0.0);
    if (f_full)
        for (int i = 0; i < d; ++i) f_free[i] = f_full[free_dofs[i]];

    gpde_vo_plan *pl = new gpde_vo_plan();   // (its VoEnv member reads the experiment switches here, once)
    pl->device = device;
    pl->n_sm = sm_count(device);
    DeviceGuard guard(device);
    VoDev &D = pl->dev;
    D.n_nodes = n_nodes; D.n_cells = n_cells; D.n_inputs = n_inputs; D.d = d; D.n_bc = n_bc; D.nslots = nslots;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = track_vo(pl, &D.ell_in, ell_in);
    if (e == cudaSuccess) e = track_vo(pl, &D.ell_j1, ell_j1);
    if (e == cudaSuccess) e = track_vo(pl, &D.ell_j2, ell_j2);
    if (e == cudaSuccess) e = track_vo(pl, &D.ell_c0, c0);
    if (e == cudaSuccess) e = track_vo(pl, &D.ell_c1, c1);
    if (e == cudaSuccess) e = track_vo(pl, &D.ell_c2, c2);
    if (e == cudaSuccess) e = track_vo(pl, &D.f_free, f_free);
    if (e == cudaSuccess) {
        std::vector<int> free_row(n_nodes), bc_row(n_nodes);
        for (int v = 0; v < n_nodes; ++v) {
            free_row[v] = src[v] >= 0 ? src[v] : -1;
            bc_row[v] = src[v] < 0 ? -src[v] - 1 : -1;
        }
        e = build_csr_terms(pl, pl->csr, d, free_row, n_cells, cell_dofs, Ke, cell_to_input, src);
        if (e == cudaSuccess) e = build_csr_terms(pl, pl->grad.bc_rows, n_bc, bc_row, n_cells, cell_dofs, Ke, cell_to_input, src);
    }
    if (e == cudaSuccess) e = build_grad_cells(pl, n_cells, cell_dofs, Ke, cell_to_input, n_inputs, src);
    if (e == cudaSuccess) e = build_fused_tiles(pl, n_nodes, n_cells, cell_dofs, Ke, cell_to_input, d, src, f_free);
    if (e != cudaSuccess) {
        gpde_vo_plan_destroy(pl);
        return fail(GPDE_ERR_CUDA, "vo_plan_create: upload failed: %s", cudaGetErrorString(e));
    }
    build_grid_plan(pl, n_nodes, n_cells, cell_dofs, Ke, cell_to_input, n_inputs, free_dofs, d, bc_dofs, n_bc, f_free);
    *plan = pl;
    return GPDE_OK;
}

int gpde_vo_plan_destroy(gpde_vo_plan *pl) {
    if (!pl) return GPDE_OK;
    DeviceGuard guard(pl->device);
    for (void *p : pl->allocs) cudaFree(p);
    delete pl;
    return GPDE_OK;
}

int gpde_vo_plan_info(const gpde_vo_plan *pl, int64_t out[8]) {
    if (!pl || !out) return fail(GPDE_ERR_ARG, "vo_plan_info: null");
    out[0] = pl->dev.n_nodes; out[1] = pl->dev.n_cells; out[2] = pl->dev.n_inputs; out[3] = pl->dev.d;
    out[4] = pl->dev.n_bc; out[5] = pl->dev.nslots; out[6] = pl->device;
    out[7] = pl->tiles.ok ? (int64_t)pl->fused_smem : 0;   // bytes of shared memory of the fused path (0 = unavailable)
    return GPDE_OK;
}

int gpde_vo_plan_kernel_path(const gpde_vo_plan *pl, int m, int elem_bytes) {
    if (!pl) return fail(GPDE_ERR_ARG, "vo_plan_kernel_path: null");
    if (use_grid(pl)) {
        Grid2Dev G;
        int NT, NX;
        size_t smem;
        if (m > 0 && m <= 32 && grid2_setup(pl, m, false, 1, G, NT, NX, smem, elem_bytes, elem_bytes)) return 2;
        if (m > 32 && grid2_setup(pl, 0, true, 1, G, NT, NX, smem, elem_bytes, elem_bytes)) return 3;
    }
    if (m > 0 && m <= 32 && use_fused(pl)) return 1;
    return 0;
}

size_t gpde_vo_workspace_bytes(const gpde_vo_plan *pl, int64_t B, int m) {
    if (!pl || B < 0) return 0;
    // version-1 kernels: K-padded rho [B][dp] + padded V [dp][ldb] (residual), V s [B][d] (residual_T)
    const size_t dp = (size_t)gemm_dp(pl->dev.d);
    // (+ up to 8 partial result tiles [B][ldb] of the split contraction)
    size_t need = sizeof(double) * (dp * (size_t)B + dp * (size_t)gemm_ldb(std::max(m, 1)) +
                                    8 * (size_t)B * (size_t)gemm_ldb(std::max(m, 1)));
    if (pl->grid.ok && m > 0) {   // residual_T on the grid path: padded s [B][mp], V^T [mp][ldb], w [B][d]
        const size_t mp = (size_t)gemm_dp(m), ldb = ((size_t)pl->dev.d + 127) / 128 * 128;
        need = std::max(need, sizeof(double) * ((size_t)B * mp + mp * ldb + (size_t)B * pl->dev.d));
    }
    if (m > 32) need = std::max(need, gridgemm_workspace_bytes(pl, (long long)B, m));
    if (pl->grid.ok && m > 0 && m <= 32) {   // packed V rows of the lean kernel (NT = 4 n-tiles: the most m <= 32 takes)
        need = std::max(need, (size_t)(pl->grid.ny + 1) * grid2_v_row_bytes(pl->grid.nx / 16, 4, 0));
        // packed V^T rows of the one-kernel transposed application (launch_grid2_wt): <= 8 k-steps
        need = std::max(need, (size_t)(pl->grid.ny + 1) * ((size_t)((pl->grid.nx + 15) / 16) * 2 * 8 * 256 + kGrid2MaskBytes));
    }
    // w = gbar_r V^T of residual_grad; a per-sample V's rho [B,d] or rows V_b s_b [B][vb_ldw] take no more than this
    if (m > 0) need = std::max(need, expand_bytes(pl, (long long)B, m));
    return need;
}

int gpde_vo_pack_weights_f64(const gpde_vo_plan *pl, const double *V, int m, int flags, void *workspace,
                             gpde_stream_t stream) {
    if (!pl || !V || !workspace) return fail(GPDE_ERR_ARG, "vo_pack_weights: null argument");
    if ((uintptr_t)workspace & 15) return fail(GPDE_ERR_ARG, "vo_pack_weights: workspace must be 16-byte aligned");
    Grid2Dev G;
    int NT, NX;
    size_t smem;
    if (!use_grid(pl) || !grid2_setup(pl, m, false, (flags & 1) ? 0 : 1, G, NT, NX, smem)) return 1;
    DeviceGuard guard(pl->device);
    grid2_pack(G, V, m, NT, NX, (double *)workspace, pl->n_sm, (cudaStream_t)stream);
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

int gpde_vo_pack_weights_f32(const gpde_vo_plan *pl, const float *V, int m, int flags, void *workspace,
                             gpde_stream_t stream) {
    if (!pl || !V || !workspace) return fail(GPDE_ERR_ARG, "vo_pack_weights: null argument");
    if ((uintptr_t)workspace & 15) return fail(GPDE_ERR_ARG, "vo_pack_weights: workspace must be 16-byte aligned");
    Grid2Dev G;
    int NT, NX;
    size_t smem;
    if (!use_grid(pl) || !grid2_setup(pl, m, false, (flags & 1) ? 0 : 1, G, NT, NX, smem, 4, 4)) return 1;
    DeviceGuard guard(pl->device);
    grid2_pack<float>(G, V, m, NT, NX, (double *)workspace, pl->n_sm, (cudaStream_t)stream);
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

int gpde_vo_posterior_f64(const gpde_vo_plan *pl, const double *a, int64_t a_stride, const double *V, int64_t v_stride,
                          int m, const double *rho, const double *noise_var, const double *g, const double *prec,
                          double *mean, double *vars, int *info, int64_t N, gpde_stream_t stream) {
    if (!pl || N < 0 || m <= 0) return fail(GPDE_ERR_ARG, "vo_posterior: bad argument");
    if (m > 64) return fail(GPDE_ERR_SIZE, "vo_posterior: m = %d > 64 weighting functions per data point", m);
    if (N == 0) return GPDE_OK;
    if (!a || !V || !rho || !noise_var || !g || !prec || !mean || !vars) return fail(GPDE_ERR_ARG, "vo_posterior: null argument");
    if (v_stride != 0 && v_stride != (int64_t)pl->dev.d * m) return fail(GPDE_ERR_ARG, "vo_posterior: v_stride must be 0 or d*m");
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (m <= 32) {
        auto kern = vo_posterior_kernel<32>;
        const size_t smem = post_smem_bytes<32>(pl->csr.max_row);
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<(unsigned)N, kPostThreads, smem, st>>>(pl->csr, a, (long long)a_stride, V, (long long)v_stride, m, rho, noise_var, g,
                                                      prec, mean, vars, info);
    } else {
        auto kern = vo_posterior_kernel<64>;
        const size_t smem = post_smem_bytes<64>(pl->csr.max_row);
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<(unsigned)N, kPostThreads, smem, st>>>(pl->csr, a, (long long)a_stride, V, (long long)v_stride, m, rho, noise_var, g,
                                                      prec, mean, vars, info);
    }
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

// Layout of the blocked posterior's workspace (vo_posterior_blocked.cuh) for N data points: row segments S of the gram pass
// so that about two waves of CTAs run (at most 8, at least 8 row tiles per segment), the same S for every data point.
static gpde::BlkLayout blocked_layout(const gpde_vo_plan *pl, long long N, int m) {
    using namespace gpde;
    BlkLayout L;
    L.mp = (m + kBlkTile - 1) / kBlkTile * kBlkTile;
    L.nb = L.mp / kBlkTile;
    L.nbt = L.nb * (L.nb + 1) / 2;
    const long long ctas = std::max(1LL, N) * L.nbt, want = 2LL * pl->n_sm;
    const int tiles = (pl->csr.d + kBlkRows - 1) / kBlkRows;
    int S = ctas >= want ? 1 : (int)((want + ctas - 1) / ctas);
    S = std::max(1, std::min({S, 8, tiles / 8}));
    L.S = S;
    L.seg = (long long)L.nbt * kBlkTile * kBlkTile + L.mp;
    L.pa = std::max((long long)S * L.seg, (long long)L.mp * L.mp);
    L.stride = L.pa + (long long)L.mp * L.mp + L.mp;
    return L;
}

size_t gpde_vo_posterior_blocked_workspace_bytes(const gpde_vo_plan *pl, int64_t N, int m) {
    if (!pl || N <= 0 || m <= 0 || m > 256) return 0;
    return sizeof(double) * (size_t)blocked_layout(pl, (long long)N, m).stride * (size_t)N;
}

int gpde_vo_posterior_blocked_f64(const gpde_vo_plan *pl, const double *a, int64_t a_stride, const double *V,
                                  int64_t v_stride, int m, const double *rho, const double *noise_var, const double *g,
                                  const double *prec, double *mean, double *vars, int *info, void *workspace,
                                  size_t workspace_bytes, int64_t N, gpde_stream_t stream) {
    if (!pl || N < 0 || m <= 0) return fail(GPDE_ERR_ARG, "vo_posterior_blocked: bad argument");
    if (m > 256) return fail(GPDE_ERR_SIZE, "vo_posterior_blocked: m = %d > 256 weighting functions per data point", m);
    if (N == 0) return GPDE_OK;
    if (!a || !V || !rho || !noise_var || !g || !prec || !mean || !vars)
        return fail(GPDE_ERR_ARG, "vo_posterior_blocked: null argument");
    if (v_stride != 0 && v_stride != (int64_t)pl->dev.d * m)
        return fail(GPDE_ERR_ARG, "vo_posterior_blocked: v_stride must be 0 or d*m");
    const size_t need = gpde_vo_posterior_blocked_workspace_bytes(pl, N, m);
    if (!workspace || ((uintptr_t)workspace & 15) || workspace_bytes < need)
        return fail(GPDE_ERR_ARG, "vo_posterior_blocked: workspace must be 16-byte aligned and hold %zu bytes", need);
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    const BlkLayout Lo = blocked_layout(pl, (long long)N, m);
    double *ws = (double *)workspace;
    const size_t sm_gram = blk_gram_smem(pl->csr.max_row), sm_factor = blk_factor_smem(Lo.mp),
                 sm_apply = blk_apply_smem(Lo.mp, pl->csr.max_row);
    GPDE_CUDA_OK(cudaFuncSetAttribute(vo_post_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_gram));
    GPDE_CUDA_OK(cudaFuncSetAttribute(vo_post_factor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_factor));
    GPDE_CUDA_OK(cudaFuncSetAttribute(vo_post_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_apply));
    vo_post_gram_kernel<<<dim3((unsigned)(Lo.nbt * Lo.S), (unsigned)N), kPostThreads, sm_gram, st>>>(
        pl->csr, a, (long long)a_stride, V, (long long)v_stride, m, rho, prec, ws, Lo);
    vo_post_factor_kernel<<<(unsigned)N, kPostThreads, sm_factor, st>>>(m, noise_var, ws, Lo, info);
    vo_post_apply_kernel<<<dim3((unsigned)((pl->csr.d + kBlkRows - 1) / kBlkRows), (unsigned)N), kPostThreads, sm_apply, st>>>(
        pl->csr, a, (long long)a_stride, V, (long long)v_stride, m, g, prec, ws, Lo, mean, vars);
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

int gpde_vo_moments_f64(const gpde_vo_plan *pl, const double *a, int64_t a_stride, const double *V, int64_t v_stride, int m,
                        const double *rho, const double *v, double *out_r, double *out_s2, int64_t N, gpde_stream_t stream) {
    if (!pl || N < 0 || m <= 0) return fail(GPDE_ERR_ARG, "vo_moments: bad argument");
    if (m > 256) return fail(GPDE_ERR_SIZE, "vo_moments: m = %d > 256 weighting functions per data point", m);
    if (N == 0) return GPDE_OK;
    if (!a || !V || !rho || !v || !out_r || !out_s2) return fail(GPDE_ERR_ARG, "vo_moments: null argument");
    if (v_stride != 0 && v_stride != (int64_t)pl->dev.d * m) return fail(GPDE_ERR_ARG, "vo_moments: v_stride must be 0 or d*m");
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (m <= 32) {
        auto kern = vo_moments_kernel<32>;
        const size_t smem = moments_smem_bytes<32>(pl->csr.max_row);
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<(unsigned)N, kPostThreads, smem, st>>>(pl->csr, a, (long long)a_stride, V, (long long)v_stride, m, rho, v, out_r, out_s2);
    } else if (m <= 64) {
        auto kern = vo_moments_kernel<64>;
        const size_t smem = moments_smem_bytes<64>(pl->csr.max_row);
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<(unsigned)N, kPostThreads, smem, st>>>(pl->csr, a, (long long)a_stride, V, (long long)v_stride, m, rho, v, out_r, out_s2);
    } else {     // one CTA per (64-column panel, data point)
        const size_t smem = blk_moments_smem(pl->csr.max_row);
        GPDE_CUDA_OK(cudaFuncSetAttribute(vo_moments_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        vo_moments_panel_kernel<<<dim3((unsigned)((m + kBlkTile - 1) / kBlkTile), (unsigned)N), kPostThreads, smem, st>>>(
            pl->csr, a, (long long)a_stride, V, (long long)v_stride, m, rho, v, out_r, out_s2);
    }
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

int gpde_vo_energy_step_f64(const gpde_vo_plan *pl, const double *a, int64_t a_stride, const double *V, int64_t v_stride,
                            int m, const double *rho, const double *g, const double *prec, const double *inv_T, double *mean,
                            int *info, int64_t N, gpde_stream_t stream) {
    if (!pl || N < 0 || m <= 0) return fail(GPDE_ERR_ARG, "vo_energy_step: bad argument");
    if (m > 64) return fail(GPDE_ERR_SIZE, "vo_energy_step: m = %d > 64 weighting functions per data point", m);
    if (N == 0) return GPDE_OK;
    if (!a || !V || !rho || !g || !prec || !inv_T || !mean) return fail(GPDE_ERR_ARG, "vo_energy_step: null argument");
    if (a_stride != 0 && a_stride != (int64_t)pl->dev.n_inputs)
        return fail(GPDE_ERR_ARG, "vo_energy_step: a_stride must be 0 or n_inputs");
    if (v_stride != 0 && v_stride != (int64_t)pl->dev.d * m) return fail(GPDE_ERR_ARG, "vo_energy_step: v_stride must be 0 or d*m");
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (m <= 32) return vo_energy_step_launch<32>(pl, a, a_stride, V, v_stride, m, rho, g, prec, inv_T, mean, info, N, st);
    return vo_energy_step_launch<64>(pl, a, a_stride, V, v_stride, m, rho, g, prec, inv_T, mean, info, N, st);
}

int gpde_vo_energy_step_blocked_f64(const gpde_vo_plan *pl, const double *a, int64_t a_stride, const double *V,
                                    int64_t v_stride, int m, const double *rho, const double *g, const double *prec,
                                    const double *inv_T, double *mean, int *info, void *workspace, size_t workspace_bytes,
                                    int64_t N, gpde_stream_t stream) {
    if (!pl || N < 0 || m <= 0) return fail(GPDE_ERR_ARG, "vo_energy_step_blocked: bad argument");
    if (m > 256) return fail(GPDE_ERR_SIZE, "vo_energy_step_blocked: m = %d > 256 weighting functions per data point", m);
    if (N == 0) return GPDE_OK;
    if (!a || !V || !rho || !g || !prec || !inv_T || !mean)
        return fail(GPDE_ERR_ARG, "vo_energy_step_blocked: null argument");
    if (a_stride != 0 && a_stride != (int64_t)pl->dev.n_inputs)
        return fail(GPDE_ERR_ARG, "vo_energy_step_blocked: a_stride must be 0 or n_inputs");
    if (v_stride != 0 && v_stride != (int64_t)pl->dev.d * m)
        return fail(GPDE_ERR_ARG, "vo_energy_step_blocked: v_stride must be 0 or d*m");
    const size_t need = gpde_vo_posterior_blocked_workspace_bytes(pl, N, m);
    if (!workspace || ((uintptr_t)workspace & 15) || workspace_bytes < need)
        return fail(GPDE_ERR_ARG, "vo_energy_step_blocked: workspace must be 16-byte aligned and hold %zu bytes", need);
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    const BlkLayout Lo = blocked_layout(pl, (long long)N, m);
    double *ws = (double *)workspace;
    void *zero_noise = nullptr;
    GPDE_CUDA_OK(cudaGetSymbolAddress(&zero_noise, energy_zero_noise));
    const size_t sm_gram = blk_gram_smem(pl->csr.max_row), sm_factor = blk_factor_smem(Lo.mp);
    GPDE_CUDA_OK(cudaFuncSetAttribute(vo_energy_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_gram));
    GPDE_CUDA_OK(cudaFuncSetAttribute(vo_post_factor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_factor));
    vo_energy_gram_kernel<<<dim3((unsigned)(Lo.nbt * Lo.S), (unsigned)N), kPostThreads, sm_gram, st>>>(
        pl->csr, a, (long long)a_stride, V, (long long)v_stride, m, rho, g, prec, inv_T, mean, ws, Lo);
    vo_post_factor_kernel<<<(unsigned)N, kPostThreads, sm_factor, st>>>(m, (const double *)zero_noise, ws, Lo, info);
    vo_energy_apply_kernel<<<dim3((unsigned)((pl->csr.d + kEnergyApplyRows - 1) / kEnergyApplyRows), (unsigned)N),
                             kPostThreads, 0, st>>>(pl->csr.d, V, (long long)v_stride, m, ws, Lo, mean);
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

int gpde_vo_residual_f64(const gpde_vo_plan *pl, const double *a, int64_t a_stride, int a_is_log, const double *y,
                         const double *g, int64_t g_stride, const double *V, int64_t v_stride, int m, double *r,
                         double *rho, void *workspace, int flags, int64_t B, gpde_stream_t stream) {
    return vo_residual<double>(pl, a, a_stride, a_is_log, y, g, g_stride, V, v_stride, m, r, rho, workspace, flags, B, stream);
}
int gpde_vo_residual_f32(const gpde_vo_plan *pl, const float *a, int64_t a_stride, int a_is_log, const float *y,
                         const float *g, int64_t g_stride, const float *V, int64_t v_stride, int m, float *r,
                         float *rho, void *workspace, int flags, int64_t B, gpde_stream_t stream) {
    return vo_residual<float>(pl, a, a_stride, a_is_log, y, g, g_stride, V, v_stride, m, r, rho, workspace, flags, B, stream);
}
int gpde_vo_residual_T_f64(const gpde_vo_plan *pl, const double *a, int64_t a_stride, int a_is_log, const double *V,
                           int64_t v_stride, int m, const double *s, double *q, void *workspace, int64_t B,
                           gpde_stream_t stream) {
    return vo_residual_T<double>(pl, a, a_stride, a_is_log, V, v_stride, m, s, q, workspace, B, stream);
}
int gpde_vo_residual_T_f32(const gpde_vo_plan *pl, const float *a, int64_t a_stride, int a_is_log, const float *V,
                           int64_t v_stride, int m, const float *s, float *q, void *workspace, int64_t B,
                           gpde_stream_t stream) {
    return vo_residual_T<float>(pl, a, a_stride, a_is_log, V, v_stride, m, s, q, workspace, B, stream);
}

int gpde_vo_residual_grad_f64(const gpde_vo_plan *pl, const double *a, int64_t a_stride, int a_is_log, const double *y,
                              const double *g, int64_t g_stride, const double *V, int64_t v_stride, int m,
                              const double *gbar_r, double *grad_a, double *grad_g, void *workspace, int64_t B,
                              gpde_stream_t stream) {
    return vo_residual_grad<double>(pl, a, a_stride, a_is_log, y, g, g_stride, V, v_stride, m, gbar_r, grad_a, grad_g,
                                    workspace, B, stream);
}
int gpde_vo_residual_grad_f32(const gpde_vo_plan *pl, const float *a, int64_t a_stride, int a_is_log, const float *y,
                              const float *g, int64_t g_stride, const float *V, int64_t v_stride, int m,
                              const float *gbar_r, float *grad_a, float *grad_g, void *workspace, int64_t B,
                              gpde_stream_t stream) {
    return vo_residual_grad<float>(pl, a, a_stride, a_is_log, y, g, g_stride, V, v_stride, m, gbar_r, grad_a, grad_g,
                                   workspace, B, stream);
}

}  // extern "C"

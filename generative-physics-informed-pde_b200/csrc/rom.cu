// Coarse-grained model on sm_100a: fused assemble -> banded LDL^T -> solve, adjoint with the
// stored factor, GetStiffness.   Replaces bottleneck/ROM.py:59-100 (+ its autograd).
//
// Maths (SURVEY.md 3.4).  With Fr/C the free/constrained dofs and x the conductivities,
//   K(x) = sum_e x_e K_e ,  K_ff u_f = F_f - K_fc g ,  u_c = g = F_c
// which is the SPD statement of the reference's "overwrite Dirichlet rows with identity rows,
// then LU" (ROM.py:97-98, :61).  K_ff is banded in the free-dof order (half bandwidth hbw), so
// the factor is a banded LDL^T (no square roots), n_f*(hbw+1) doubles per sample, held in shared
// memory while it is used and stashed once for the adjoint.
//
// Work decomposition: G lanes (8/16/32, chosen from the band window size) own one sample; a CTA
// of 4 warps owns 4*32/G samples.  Per elimination step the hbw(hbw+1)/2 window updates are
// spread over the G lanes and the forward substitution rides along as an extra column, so a
// step costs one __syncwarp.
#include "common.cuh"

#include <algorithm>
#include <cmath>

namespace gpde {
thread_local char g_last_error[512] = "";

struct RomDev {
    int n, E, n_bc, n_free, hbw, bw1, n_band, n_pairs;
    const int *free_dof;   // [n_free]  free-local -> dof
    const int *bc_dof;     // [n_bc]
    // band assembly: Ab[p] = sum_t band_coef[t] * x[band_elem[t]],  p = i*bw1 + (i-j)
    const int *band_ptr, *band_elem;
    const double *band_coef;
    // rhs coupling: z[i] = F[free_i] - sum_t rhs_coef[t] * x[rhs_elem[t]] * F[rhs_dof[t]]
    const int *rhs_ptr, *rhs_elem, *rhs_dof;
    const double *rhs_coef;
    // gradient: gx[e] = - sum_t grad_coef[t] * lam[grad_i[t]] * u[grad_j[t]]   (grad_i free-local)
    const int *grad_ptr, *grad_i, *grad_j;
    const double *grad_coef;
    // constrained rows of lambda: lam_c = gbar_c - sum_t cf_coef[t] * x[cf_elem[t]] * lam[cf_free[t]]
    const int *cf_ptr, *cf_elem, *cf_free;
    const double *cf_coef;
    // window pair table, ordered so that a window of w rows uses the first w(w+1)/2 pairs
    const unsigned char *pair_si, *pair_sj;
    // dense stiffness (GetStiffness): entry ij -> list of (elem, coef)
    const int *st_ptr, *st_elem;
    const double *st_coef;
    const unsigned char *is_bc;  // [n]
    // every table the forward / adjoint kernels read lives in ONE device arena (st_* excluded); the kernels
    // copy it into shared memory once per CTA and read the tables there (no dependent global loads)
    const char *arena;
    int arena_bytes;
};

constexpr int kRomThreads = 128;

__device__ __forceinline__ double ld_as_double(const double *p) { return *p; }
__device__ __forceinline__ double ld_as_double(const float *p) { return (double)*p; }

// 1/d for a positive, finite pivot: hardware seed + two Newton steps (<= 1 ulp; the IEEE division sequence is
// ~4x the instructions and sits on the critical path of every elimination step)
__device__ __forceinline__ double fast_rcp(double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    r = fma(r, fma(-d, r, 1.0), r);
    r = fma(r, fma(-d, r, 1.0), r);
    return r;
}
}  // namespace gpde

#include "rom_tps.cuh"
#include "rom_tpw.cuh"

struct gpde_rom_plan {
    gpde::RomDev dev;
    int device;
    int tps;                // 1: the thread-per-sample kernels (rom_tps.cuh) serve this plan (no factor stash)
    gpde::TpsAdjTab<gpde::TpsShape4x4> tps_tab;   // their tables, passed by value with every launch
    int tpw;                // 1: the windowed thread-per-sample kernels (rom_tpw.cuh); the factor stash is sample-interleaved
    const gpde::TpwFwdTab<gpde::TpwShape8x8> *tpw_fwd;   // their tables, in device memory (each CTA copies them to shared memory)
    const gpde::TpwAdjTab<gpde::TpwShape8x8> *tpw_adj;
    int lanes;              // G
    int n_contrib;
    size_t smem_fwd, smem_adj;  // bytes per sample
    std::vector<void *> allocs;
};

namespace gpde {

// ---------------------------------------------------------------------------------------------
// Shared building blocks (all called by the G lanes of one sample, converged).
// ---------------------------------------------------------------------------------------------
template <typename T, int G>
__device__ __forceinline__ int load_conductivities(const RomDev &P, const T *__restrict__ X, int x_is_log,
                                                   long long b, int gl, double *xs, double *dxs) {
    int bad = 0;
    for (int e = gl; e < P.E; e += G) {
        double v = ld_as_double(X + b * P.E + e);
        double dv = 1.0;
        if (x_is_log) {   // components.py:298  x = exp(X) + 1e-8
            dv = exp(v);
            v = dv + 1e-8;
        }
        if (!(v > 1e-12)) bad = GPDE_INFO_NONPOSITIVE_X;   // ROM.py:74-76
        xs[e] = v;
        if (dxs) dxs[e] = dv;
    }
    return bad;
}

template <int G>
__device__ __forceinline__ void assemble_band(const RomDev &P, int gl, const double *xs, double *Ab) {
    for (int p = gl; p < P.n_band; p += G) {
        double acc = 0.0;
        const int t1 = P.band_ptr[p + 1];
        for (int t = P.band_ptr[p]; t < t1; ++t) acc = fma(P.band_coef[t], xs[P.band_elem[t]], acc);
        Ab[p] = acc;
    }
}

// In-place banded LDL^T of Ab (column entries stay unscaled: Ab[(k+s)*bw1+s] = l_{k+s,k} d_k),
// dinv[k] = 1/d_k.  If z != nullptr the forward substitution w = D^-1 L^-1 z rides along.
template <int G>
__device__ __forceinline__ int factor_band(const RomDev &P, int gl, double *Ab, double *dinv, double *z,
                                           double *wv) {
    int bad = 0;
    const int bw1 = P.bw1, nf = P.n_free, hbw = P.hbw;
    for (int k = 0; k < nf; ++k) {
        const double d = Ab[k * bw1];
        if (!(d > 0.0)) bad = GPDE_INFO_NOT_SPD;
        const double invd = fast_rcp(d);
        const int wlen = min(hbw, nf - 1 - k);
        const int npairs = (wlen * (wlen + 1)) >> 1;
        for (int q = gl; q < npairs; q += G) {
            const int si = P.pair_si[q], sj = P.pair_sj[q];
            const double ci = Ab[(k + si) * bw1 + si];
            const double cj = Ab[(k + sj) * bw1 + sj];
            // scaled before the product: ci * cj overflows once the entries pass ~1e154 (conductivities up to exp(709))
            Ab[(k + si) * bw1 + (si - sj)] -= ci * (cj * invd);
        }
        if (z) {
            const double wk = z[k] * invd;
            for (int s = gl + 1; s <= wlen; s += G) z[k + s] -= Ab[(k + s) * bw1 + s] * wk;
            if (gl == 0) wv[k] = wk;
        }
        if (gl == 0) dinv[k] = invd;
        __syncwarp();
    }
    return bad;
}

// w = D^-1 L^-1 z with a stored factor (z is consumed).
template <int G>
__device__ __forceinline__ void forward_subst(const RomDev &P, int gl, const double *Ab, const double *dinv,
                                              double *z, double *wv) {
    const int bw1 = P.bw1, nf = P.n_free, hbw = P.hbw;
    for (int k = 0; k < nf; ++k) {
        const double wk = z[k] * dinv[k];
        const int wlen = min(hbw, nf - 1 - k);
        for (int s = gl + 1; s <= wlen; s += G) z[k + s] -= Ab[(k + s) * bw1 + s] * wk;
        if (gl == 0) wv[k] = wk;
        __syncwarp();
    }
}

// Solves L^T sol = w (unit-lower L = column entries * dinv).  acc is scratch [n_free].
// sol_k = w_k - dinv_k * sum_{s>=1} Ab[(k+s)*bw1+s] sol_{k+s}; written to out[out_index[k]].
template <int G>
__device__ __forceinline__ void backward_subst(const RomDev &P, int gl, const double *Ab, const double *dinv,
                                               const double *wv, double *acc, double *out,
                                               const int *__restrict__ out_index) {
    const int bw1 = P.bw1, nf = P.n_free, hbw = P.hbw;
    for (int i = gl; i < nf; i += G) acc[i] = 0.0;
    __syncwarp();
    for (int k = nf - 1; k >= 0; --k) {
        const double sk = wv[k] - dinv[k] * acc[k];
        const int wlen = min(hbw, k);
        for (int s = gl + 1; s <= wlen; s += G) acc[k - s] = fma(Ab[k * bw1 + s], sk, acc[k - s]);
        if (gl == 0) out[out_index ? out_index[k] : k] = sk;
        __syncwarp();
    }
}


// Copies the plan's table arena into shared memory (once per CTA) and returns a RomDev whose table pointers
// point at the copy.  sample_smem is set to the first 16-byte aligned address after it.
__device__ __forceinline__ RomDev stage_tables(const RomDev &P, double *smem, double **sample_smem) {
    char *dst = reinterpret_cast<char *>(smem);
    const uint4 *src = reinterpret_cast<const uint4 *>(P.arena);
    for (int i = threadIdx.x; i < P.arena_bytes / 16; i += blockDim.x) reinterpret_cast<uint4 *>(dst)[i] = src[i];
    __syncthreads();
    RomDev Q = P;
    // derive the new pointers from the shared-memory base (not from the kernel-parameter pointers, which the
    // compiler knows to be global and would keep loading with ld.global)
#define GPDE_REBASE(f) \
    Q.f = reinterpret_cast<decltype(Q.f)>(dst + (size_t)(reinterpret_cast<const char *>(P.f) - P.arena))
    GPDE_REBASE(free_dof); GPDE_REBASE(bc_dof);
    GPDE_REBASE(band_ptr); GPDE_REBASE(band_elem); GPDE_REBASE(band_coef);
    GPDE_REBASE(rhs_ptr); GPDE_REBASE(rhs_elem); GPDE_REBASE(rhs_dof); GPDE_REBASE(rhs_coef);
    GPDE_REBASE(grad_ptr); GPDE_REBASE(grad_i); GPDE_REBASE(grad_j); GPDE_REBASE(grad_coef);
    GPDE_REBASE(cf_ptr); GPDE_REBASE(cf_elem); GPDE_REBASE(cf_free); GPDE_REBASE(cf_coef);
    GPDE_REBASE(pair_si); GPDE_REBASE(pair_sj);
#undef GPDE_REBASE
    *sample_smem = smem + P.arena_bytes / 8;
    return Q;
}

// ---------------------------------------------------------------------------------------------
// forward:  X, F -> u (+ factor stash)
// ---------------------------------------------------------------------------------------------
template <typename T, int G>
__global__ void __launch_bounds__(kRomThreads)
rom_forward_kernel(RomDev P0, const T *__restrict__ X, int x_is_log, const T *__restrict__ F,
                   T *__restrict__ u, double *__restrict__ factor, int *info, long long B,
                   int smem_doubles_per_sample) {
    extern __shared__ __align__(16) double smem_all[];
    double *smem;
    const RomDev P = stage_tables(P0, smem_all, &smem);
    constexpr int GPW = 32 / G;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gl = lane % G, gidx = warp * GPW + lane / G;
    const int groups_per_block = (kRomThreads / 32) * GPW;
    long long b = (long long)blockIdx.x * groups_per_block + gidx;
    const bool active = b < B;
    if (!active) b = B - 1;

    double *xs = smem + (size_t)gidx * smem_doubles_per_sample;   // [E]
    double *Fs = xs + P.E;                                           // [n]   F, then u
    double *Ab = Fs + P.n;                                           // [n_band]
    double *z = Ab + P.n_band;                                       // [n_free]
    double *wv = z + P.n_free;                                       // [n_free]
    double *dinv = wv + P.n_free;                                    // [n_free]

    int bad = load_conductivities<T, G>(P, X, x_is_log, b, gl, xs, nullptr);
    for (int i = gl; i < P.n; i += G) Fs[i] = ld_as_double(F + b * P.n + i);
    __syncwarp();

    assemble_band<G>(P, gl, xs, Ab);
    for (int i = gl; i < P.n_free; i += G) {
        double acc = Fs[P.free_dof[i]];
        const int t1 = P.rhs_ptr[i + 1];
        for (int t = P.rhs_ptr[i]; t < t1; ++t)
            acc -= P.rhs_coef[t] * xs[P.rhs_elem[t]] * Fs[P.rhs_dof[t]];
        z[i] = acc;
    }
    __syncwarp();

    bad |= factor_band<G>(P, gl, Ab, dinv, z, wv);
    backward_subst<G>(P, gl, Ab, dinv, wv, z, Fs, P.free_dof);

    if (factor) {   // uniform branch: every lane of the warp reaches the barrier, the stores are predicated per sample
        double *fb = factor + b * (long long)P.n_band;
        // band entries as they are; the diagonal slots then receive 1/d_k (no index divisions)
        if (active)
            for (int p = gl; p < P.n_band; p += G) fb[p] = Ab[p];
        __syncwarp();
        if (active)
            for (int k = gl; k < P.n_free; k += G) fb[k * P.bw1] = dinv[k];
    }
    if (active) {
        for (int i = gl; i < P.n; i += G) u[b * P.n + i] = (T)Fs[i];
        if (bad && info) atomicOr(info, bad);
    }
}

// ---------------------------------------------------------------------------------------------
// adjoint:  gbar_u -> gradX (, gradF)
// ---------------------------------------------------------------------------------------------
template <typename T, int G>
__global__ void __launch_bounds__(kRomThreads)
rom_adjoint_kernel(RomDev P0, const T *__restrict__ X, int x_is_log, const T *__restrict__ u,
                   const double *__restrict__ factor, const T *__restrict__ gbar, T *__restrict__ gradX,
                   T *__restrict__ gradF, long long B, int smem_doubles_per_sample) {
    extern __shared__ __align__(16) double smem_all[];
    double *smem;
    const RomDev P = stage_tables(P0, smem_all, &smem);
    constexpr int GPW = 32 / G;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gl = lane % G, gidx = warp * GPW + lane / G;
    const int groups_per_block = (kRomThreads / 32) * GPW;
    long long b = (long long)blockIdx.x * groups_per_block + gidx;
    const bool active = b < B;
    if (!active) b = B - 1;

    double *xs = smem + (size_t)gidx * smem_doubles_per_sample;   // [E]
    double *dxs = xs + P.E;                                          // [E]
    double *us = dxs + P.E;                                          // [n]
    double *gs = us + P.n;                                           // [n]
    double *Ab = gs + P.n;                                           // [n_band]
    double *z = Ab + P.n_band;                                       // [n_free]
    double *wv = z + P.n_free;                                       // [n_free]
    double *dinv = wv + P.n_free;                                    // [n_free]
    double *lam = dinv + P.n_free;                                   // [n_free]

    load_conductivities<T, G>(P, X, x_is_log, b, gl, xs, dxs);
    for (int i = gl; i < P.n; i += G) {
        us[i] = ld_as_double(u + b * P.n + i);
        gs[i] = ld_as_double(gbar + b * P.n + i);
    }
    if (factor) {
        const double *fb = factor + b * (long long)P.n_band;
        for (int p = gl; p < P.n_band; p += G) Ab[p] = fb[p];
        for (int k = gl; k < P.n_free; k += G) dinv[k] = fb[k * P.bw1];
    }
    __syncwarp();
    if (!factor) {
        assemble_band<G>(P, gl, xs, Ab);
        __syncwarp();
        factor_band<G>(P, gl, Ab, dinv, nullptr, nullptr);
    }
    for (int i = gl; i < P.n_free; i += G) z[i] = gs[P.free_dof[i]];
    __syncwarp();
    forward_subst<G>(P, gl, Ab, dinv, z, wv);
    backward_subst<G>(P, gl, Ab, dinv, wv, z, lam, nullptr);

    if (active) {
        for (int e = gl; e < P.E; e += G) {
            double acc = 0.0;
            const int t1 = P.grad_ptr[e + 1];
            for (int t = P.grad_ptr[e]; t < t1; ++t)
                acc = fma(P.grad_coef[t] * lam[P.grad_i[t]], us[P.grad_j[t]], acc);
            gradX[b * P.E + e] = (T)(-acc * dxs[e]);
        }
        if (gradF) {
            for (int i = gl; i < P.n_free; i += G) gradF[b * P.n + P.free_dof[i]] = (T)lam[i];
            for (int c = gl; c < P.n_bc; c += G) {
                double acc = gs[P.bc_dof[c]];
                const int t1 = P.cf_ptr[c + 1];
                for (int t = P.cf_ptr[c]; t < t1; ++t)
                    acc -= P.cf_coef[t] * xs[P.cf_elem[t]] * lam[P.cf_free[t]];
                gradF[b * P.n + P.bc_dof[c]] = (T)acc;
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------
// GetStiffness: K[n,n,B] (batch last, ROM.py:93), Dirichlet rows -> identity rows (:97-98)
// ---------------------------------------------------------------------------------------------
__global__ void rom_stiffness_kernel(RomDev P, const double *__restrict__ X, double *__restrict__ K,
                                     int dirichlet, long long B) {
    const long long total = (long long)P.n * P.n * B;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long ij = idx / B, b = idx - ij * B;
        const int i = (int)(ij / P.n), j = (int)(ij - (long long)i * P.n);
        double acc = 0.0;
        if (dirichlet && P.is_bc[i]) {
            acc = (i == j) ? 1.0 : 0.0;
        } else {
            const int t1 = P.st_ptr[ij + 1];
            for (int t = P.st_ptr[ij]; t < t1; ++t) acc = fma(P.st_coef[t], X[b * P.E + P.st_elem[t]], acc);
        }
        K[idx] = acc;
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// Tables of the thread-per-sample kernels for shape S; false if M does not fit the shape (sizes, bandwidth, or more
// terms per entry than the shape provides): the plan then stays on the cooperative kernels.
template <class S>
static bool build_tps_tables(int n, int E, int nf, int hbw, const std::vector<int> &free_dof, const std::vector<int> &bc_dof,
                             const std::vector<unsigned char> &is_bc, const double *M, TpsAdjTab<S> &A) {
    if (n != S::N || E != S::E || nf != S::NF || hbw != S::HBW) return false;
    static_assert(S::N <= S::E, "the adjoint kernel stages u into the columns of x");
    static_assert(S::E * kTpsPitch < 65536 && S::N * kTpsPitch < 65536, "column offsets are 16-bit");
    auto Mat = [&](int i, int j, int e) { return M[((size_t)i * n + j) * E + e]; };
    memset(&A, 0, sizeof(A));
    TpsFwdTab<S> &Ft = A.f;
    for (int i = 0; i < nf; ++i) {
        Ft.free_dof[i] = (unsigned short)(free_dof[i] * kTpsPitch);
        int cnt = 0;
        for (int e = 0; e < E; ++e) {
            const double v = Mat(free_dof[i], free_dof[i], e);
            if (v == 0.0) continue;
            if (cnt == S::TD) return false;
            Ft.diag_coef[i * S::TD + cnt] = v;
            Ft.diag_elem[i * S::TD + cnt] = (unsigned short)(e * kTpsPitch);
            ++cnt;
        }
        for (int s = 1; s <= hbw && s <= i; ++s) {
            cnt = 0;
            for (int e = 0; e < E; ++e) {
                const double v = Mat(free_dof[i], free_dof[i - s], e);
                if (v == 0.0) continue;
                if (cnt == S::TO) return false;
                const int k = (i * S::HBW + s - 1) * S::TO + cnt;
                Ft.off_coef[k] = v;
                Ft.off_elem[k] = (unsigned short)(e * kTpsPitch);
                ++cnt;
            }
        }
        cnt = 0;
        for (size_t c = 0; c < bc_dof.size(); ++c)
            for (int e = 0; e < E; ++e) {
                const double v = Mat(free_dof[i], bc_dof[c], e);
                if (v == 0.0) continue;
                if (cnt == S::TR) return false;
                const int k = i * S::TR + cnt;
                Ft.rhs_coef[k] = v;
                Ft.rhs_elem[k] = (unsigned short)(e * kTpsPitch);
                Ft.rhs_dof[k] = (unsigned short)(bc_dof[c] * kTpsPitch);
                ++cnt;
            }
    }
    for (int e = 0; e < E; ++e) {
        int cnt = 0;
        for (int i = 0; i < n; ++i) {
            if (is_bc[i]) continue;   // overwritten rows contribute nothing (SURVEY.md 3.4)
            for (int j = 0; j < n; ++j) {
                const double v = Mat(i, j, e);
                if (v == 0.0) continue;
                if (cnt == S::TG) return false;
                const int k = e * S::TG + cnt;
                A.grad_coef[k] = v;
                A.grad_i[k] = (unsigned short)(i * kTpsPitch);
                A.grad_j[k] = (unsigned short)(j * kTpsPitch);
                ++cnt;
            }
        }
    }
    return true;
}

// Tables of the windowed thread-per-sample kernels (rom_tpw.cuh) for shape S; false if M does not fit: sizes, bandwidth,
// more terms per entry than the shape provides, or a structural non-zero inside the band other than s = 1 and s = HBW.
template <class S>
static bool build_tpw_tables(int n, int E, int nf, int hbw, const std::vector<int> &free_dof, const std::vector<int> &bc_dof,
                             const std::vector<unsigned char> &is_bc, const double *M, TpwFwdTab<S> &Ft, TpwAdjTab<S> &At) {
    if (n != S::N || E != S::E || nf != S::NF || hbw != S::HBW) return false;
    static_assert(S::E * kTpwPitch < 65536 && (S::N + 1) * kTpwPitch < 65536, "column offsets are 16-bit");
    auto Mat = [&](int i, int j, int e) { return M[((size_t)i * n + j) * E + e]; };
    memset(&Ft, 0, sizeof(Ft));
    memset(&At, 0, sizeof(At));
    for (int i = 0; i < nf; ++i) {
        TpwRow<S> &R = Ft.row[i];
        R.free_dof = At.free_dof[i] = (unsigned short)(free_dof[i] * kTpwPitch);
        int cnt = 0;
        for (int e = 0; e < E; ++e) {
            const double v = Mat(free_dof[i], free_dof[i], e);
            if (v == 0.0) continue;
            if (cnt == S::TD) return false;
            R.diag_coef[cnt] = v;
            R.diag_elem[cnt] = (unsigned short)(e * kTpwPitch);
            ++cnt;
        }
        for (int s = 1; s <= hbw && s <= i; ++s) {
            cnt = 0;
            for (int e = 0; e < E; ++e) {
                const double v = Mat(free_dof[i], free_dof[i - s], e);
                if (v == 0.0) continue;
                if (s != 1 && s != hbw) return false;       // not the 5-point structure
                if (cnt == S::TO) return false;
                double *coef = s == 1 ? R.s1_coef : R.sh_coef;
                unsigned short *elem = s == 1 ? R.s1_elem : R.sh_elem;
                coef[cnt] = v;
                elem[cnt] = (unsigned short)(e * kTpwPitch);
                ++cnt;
            }
        }
        cnt = 0;
        for (size_t c = 0; c < bc_dof.size(); ++c)
            for (int e = 0; e < E; ++e) {
                const double v = Mat(free_dof[i], bc_dof[c], e);
                if (v == 0.0) continue;
                if (cnt == S::TR) return false;
                const int k = i * S::TR + cnt;
                R.rhs_coef[cnt] = At.rhs_coef[k] = v;
                R.rhs_elem[cnt] = (unsigned short)(e * kTpwPitch);
                At.rhs_elem[k] = (unsigned short)e;
                R.rhs_dof[cnt] = At.rhs_dof[k] = (unsigned short)(bc_dof[c] * kTpwPitch);
                ++cnt;
            }
    }
    // gradient in edge form (rom_tpw.cuh): every element matrix must be symmetric with zero row sums
    for (int e = 0; e < E; ++e) {
        std::vector<int> verts;
        for (int i = 0; i < n; ++i) {
            bool used = false;
            for (int j = 0; j < n; ++j)
                if (Mat(i, j, e) != 0.0 || Mat(j, i, e) != 0.0) used = true;
            if (used) verts.push_back(i);
        }
        double scale = 0.0;
        for (int i : verts)
            for (int j : verts) scale = std::max(scale, std::fabs(Mat(i, j, e)));
        const double tol = 1e-12 * scale;
        int cnt = 0;
        for (size_t a = 0; a < verts.size(); ++a) {
            double rs = 0.0;
            for (size_t b = 0; b < verts.size(); ++b) {
                rs += Mat(verts[a], verts[b], e);
                if (std::fabs(Mat(verts[a], verts[b], e) - Mat(verts[b], verts[a], e)) > tol) return false;
            }
            if (std::fabs(rs) > 1e-9 * scale) return false;
            for (size_t b = a + 1; b < verts.size(); ++b) {
                const double w = -Mat(verts[a], verts[b], e);
                if (w == 0.0) continue;
                if (cnt == kTpwEdges) return false;
                const int k = e * kTpwEdges + cnt;
                At.edge_w[k] = w;
                const int va = verts[a], vb = verts[b];
                At.lam_a[k] = (unsigned short)((is_bc[va] ? n : va) * kTpwPitch);     // column n of the lambda array holds zeros
                At.lam_b[k] = (unsigned short)((is_bc[vb] ? n : vb) * kTpwPitch);
                At.u_a[k] = (unsigned short)(va * kTpwPitch);
                At.u_b[k] = (unsigned short)(vb * kTpwPitch);
                ++cnt;
            }
        }
    }
    return true;
}

template <typename T>
static int track(gpde_rom_plan *pl, const T **dst, const std::vector<T> &src) {
    T *p = nullptr;
    GPDE_CUDA_OK(upload(&p, src));
    pl->allocs.push_back((void *)p);
    *dst = p;
    return GPDE_OK;
}

template <typename T, int G>
static int launch_forward(const gpde_rom_plan *pl, const T *X, int x_is_log, const T *F, T *u, double *factor,
                          int *info, int64_t B, cudaStream_t st) {
    const int groups = (kRomThreads / 32) * (32 / G);
    const int per = (int)(pl->smem_fwd / sizeof(double));
    const size_t smem = (size_t)groups * pl->smem_fwd + (size_t)pl->dev.arena_bytes;
    auto kern = rom_forward_kernel<T, G>;
    GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long grid = (B + groups - 1) / groups;
    kern<<<(unsigned)grid, kRomThreads, smem, st>>>(pl->dev, X, x_is_log, F, u, factor, info, B, per);
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

template <typename T, int G>
static int launch_adjoint(const gpde_rom_plan *pl, const T *X, int x_is_log, const T *u, const double *factor,
                          const T *gbar, T *gradX, T *gradF, int64_t B, cudaStream_t st) {
    const int groups = (kRomThreads / 32) * (32 / G);
    const int per = (int)(pl->smem_adj / sizeof(double));
    const size_t smem = (size_t)groups * pl->smem_adj + (size_t)pl->dev.arena_bytes;
    auto kern = rom_adjoint_kernel<T, G>;
    GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long grid = (B + groups - 1) / groups;
    kern<<<(unsigned)grid, kRomThreads, smem, st>>>(pl->dev, X, x_is_log, u, factor, gbar, gradX, gradF, B, per);
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

template <typename T>
static int rom_forward(const gpde_rom_plan *pl, const T *X, int x_is_log, const T *F, T *u, double *factor,
                       int *info, int64_t B, gpde_stream_t stream) {
    if (!pl || B < 0) return fail(GPDE_ERR_ARG, "rom_forward: null plan or negative batch");
    if (B == 0) return GPDE_OK;
    if (!X || !F || !u) return fail(GPDE_ERR_ARG, "rom_forward: null argument");
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (pl->tps) {   // thread per sample, no factor stash (``factor`` is not touched)
        using S = TpsShape4x4;
        auto kern = rom_tps_forward_kernel<T, S>;
        constexpr size_t smem = tps_smem_forward<S>();
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<(unsigned)((B + kTpsThreads - 1) / kTpsThreads), kTpsThreads, smem, st>>>(pl->tps_tab.f, X, x_is_log, F, u, info, B);
        GPDE_CUDA_OK(cudaGetLastError());
        return GPDE_OK;
    }
    if (pl->tpw && factor) {   // thread per sample, band streamed through a register window: the kernel itself streams the
                               // factor through the stash (without one the cooperative kernels below serve the call)
        using S = TpwShape8x8;
        auto kern = rom_tpw_forward_kernel<T, S>;
        constexpr size_t smem = tpw_smem_forward<S>();
        GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<(unsigned)((B + kTpwThreads - 1) / kTpwThreads), kTpwThreads, smem, st>>>(pl->tpw_fwd, X, x_is_log, F, u, factor, info, B);
        GPDE_CUDA_OK(cudaGetLastError());
        return GPDE_OK;
    }
    switch (pl->lanes) {
        case 8: return launch_forward<T, 8>(pl, X, x_is_log, F, u, factor, info, B, st);
        case 16: return launch_forward<T, 16>(pl, X, x_is_log, F, u, factor, info, B, st);
        default: return launch_forward<T, 32>(pl, X, x_is_log, F, u, factor, info, B, st);
    }
}

template <typename T>
static int rom_adjoint(const gpde_rom_plan *pl, const T *X, int x_is_log, const T *u, const double *factor,
                       const T *gbar, T *gradX, T *gradF, int64_t B, gpde_stream_t stream) {
    if (!pl || B < 0) return fail(GPDE_ERR_ARG, "rom_adjoint: null plan or negative batch");
    if (B == 0) return GPDE_OK;
    if (!X || !u || !gbar || !gradX) return fail(GPDE_ERR_ARG, "rom_adjoint: null argument");
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (pl->tps) {   // re-assembles and re-factorises: cheaper than a factor round trip through HBM at this size
        using S = TpsShape4x4;
        const unsigned grid = (unsigned)((B + kTpsThreads - 1) / kTpsThreads);
        if (gradF) {
            auto kern = rom_tps_adjoint_kernel<T, S, true>;
            constexpr size_t smem = tps_smem_adjoint<S>(true);
            GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<grid, kTpsThreads, smem, st>>>(pl->tps_tab, X, x_is_log, u, gbar, gradX, gradF, B);
        } else {
            auto kern = rom_tps_adjoint_kernel<T, S, false>;
            constexpr size_t smem = tps_smem_adjoint<S>(false);
            GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<grid, kTpsThreads, smem, st>>>(pl->tps_tab, X, x_is_log, u, gbar, gradX, gradF, B);
        }
        GPDE_CUDA_OK(cudaGetLastError());
        return GPDE_OK;
    }
    if (pl->tpw && factor) {   // (no stash: the cooperative adjoint below re-factorises)
        using S = TpwShape8x8;
        const unsigned grid = (unsigned)((B + kTpwThreads - 1) / kTpwThreads);
        constexpr size_t smem = tpw_smem_adjoint<S>();
        if (gradF) {
            auto kern = rom_tpw_adjoint_kernel<T, S, true>;
            GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<grid, kTpwThreads, smem, st>>>(pl->tpw_adj, X, x_is_log, u, factor, gbar, gradX, gradF, B);
        } else {
            auto kern = rom_tpw_adjoint_kernel<T, S, false>;
            GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            kern<<<grid, kTpwThreads, smem, st>>>(pl->tpw_adj, X, x_is_log, u, factor, gbar, gradX, gradF, B);
        }
        GPDE_CUDA_OK(cudaGetLastError());
        return GPDE_OK;
    }
    switch (pl->lanes) {
        case 8: return launch_adjoint<T, 8>(pl, X, x_is_log, u, factor, gbar, gradX, gradF, B, st);
        case 16: return launch_adjoint<T, 16>(pl, X, x_is_log, u, factor, gbar, gradX, gradF, B, st);
        default: return launch_adjoint<T, 32>(pl, X, x_is_log, u, factor, gbar, gradX, gradF, B, st);
    }
}

}  // namespace gpde

using namespace gpde;

extern "C" {

int gpde_version(void) { return 101; }
const char *gpde_last_error(void) { return gpde::g_last_error; }

int gpde_rom_plan_create(gpde_rom_plan **plan, int n, int E, const double *M, const int64_t *bc_dofs, int n_bc,
                         int device) {
    if (!plan || !M || n <= 0 || E <= 0 || n_bc < 0 || (n_bc > 0 && !bc_dofs))
        return fail(GPDE_ERR_ARG, "rom_plan_create: bad argument");
    std::vector<unsigned char> is_bc(n, 0);
    for (int c = 0; c < n_bc; ++c) {
        if (bc_dofs[c] < 0 || bc_dofs[c] >= n) return fail(GPDE_ERR_ARG, "rom_plan_create: bc dof out of range");
        is_bc[bc_dofs[c]] = 1;
    }
    std::vector<int> free_dof, bc_dof, free_local(n, -1);
    for (int i = 0; i < n; ++i) {
        if (is_bc[i]) bc_dof.push_back(i);
        else {
            free_local[i] = (int)free_dof.size();
            free_dof.push_back(i);
        }
    }
    const int nf = (int)free_dof.size();
    if (nf == 0) return fail(GPDE_ERR_ARG, "rom_plan_create: no free dofs");
    std::vector<int> bc_local(n, -1);
    for (size_t c = 0; c < bc_dof.size(); ++c) bc_local[bc_dof[c]] = (int)c;

    auto Mat = [&](int i, int j, int e) { return M[((size_t)i * n + j) * E + e]; };

    // half bandwidth of K_ff in free-local order (exact zeros dropped)
    int hbw = 0;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            if (is_bc[i] || is_bc[j]) continue;
            for (int e = 0; e < E; ++e)
                if (Mat(i, j, e) != 0.0) {
                    hbw = std::max(hbw, std::abs(free_local[i] - free_local[j]));
                    break;
                }
        }
    if (hbw > 255) return fail(GPDE_ERR_SIZE, "rom_plan_create: half bandwidth %d > 255", hbw);
    const int bw1 = hbw + 1, n_band = nf * bw1;

    std::vector<int> band_ptr(n_band + 1, 0), band_elem;
    std::vector<double> band_coef;
    for (int i = 0; i < nf; ++i)
        for (int s = 0; s <= hbw; ++s) {
            const int p = i * bw1 + s, j = i - s;
            if (j >= 0) {
                // symmetrised entry: the reference solves with K as assembled; K_e are symmetric
                for (int e = 0; e < E; ++e) {
                    const double v = Mat(free_dof[i], free_dof[j], e);
                    if (v != 0.0) {
                        band_elem.push_back(e);
                        band_coef.push_back(v);
                    }
                }
            }
            band_ptr[p + 1] = (int)band_elem.size();
        }
    std::vector<int> rhs_ptr(nf + 1, 0), rhs_elem, rhs_dof;
    std::vector<double> rhs_coef;
    for (int i = 0; i < nf; ++i) {
        for (size_t c = 0; c < bc_dof.size(); ++c)
            for (int e = 0; e < E; ++e) {
                const double v = Mat(free_dof[i], bc_dof[c], e);
                if (v != 0.0) {
                    rhs_elem.push_back(e);
                    rhs_dof.push_back(bc_dof[c]);
                    rhs_coef.push_back(v);
                }
            }
        rhs_ptr[i + 1] = (int)rhs_elem.size();
    }
    std::vector<int> grad_ptr(E + 1, 0), grad_i, grad_j;
    std::vector<double> grad_coef;
    for (int e = 0; e < E; ++e) {
        for (int i = 0; i < n; ++i) {
            if (is_bc[i]) continue;   // overwritten rows contribute nothing (SURVEY.md 3.4)
            for (int j = 0; j < n; ++j) {
                const double v = Mat(i, j, e);
                if (v != 0.0) {
                    grad_i.push_back(free_local[i]);
                    grad_j.push_back(j);
                    grad_coef.push_back(v);
                }
            }
        }
        grad_ptr[e + 1] = (int)grad_i.size();
    }
    // lambda on constrained rows: A^T lambda = gbar, columns c of A hold K[f,c] for free rows f
    std::vector<int> cf_ptr(bc_dof.size() + 1, 0), cf_elem, cf_free;
    std::vector<double> cf_coef;
    for (size_t c = 0; c < bc_dof.size(); ++c) {
        for (int f = 0; f < nf; ++f)
            for (int e = 0; e < E; ++e) {
                const double v = Mat(free_dof[f], bc_dof[c], e);
                if (v != 0.0) {
                    cf_elem.push_back(e);
                    cf_free.push_back(f);
                    cf_coef.push_back(v);
                }
            }
        cf_ptr[c + 1] = (int)cf_elem.size();
    }
    std::vector<unsigned char> pair_si, pair_sj;
    for (int si = 1; si <= hbw; ++si)
        for (int sj = 1; sj <= si; ++sj) {
            pair_si.push_back((unsigned char)si);
            pair_sj.push_back((unsigned char)sj);
        }
    std::vector<int> st_ptr((size_t)n * n + 1, 0), st_elem;
    std::vector<double> st_coef;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            for (int e = 0; e < E; ++e) {
                const double v = Mat(i, j, e);
                if (v != 0.0) {
                    st_elem.push_back(e);
                    st_coef.push_back(v);
                }
            }
            st_ptr[(size_t)i * n + j + 1] = (int)st_elem.size();
        }

    gpde_rom_plan *pl = new gpde_rom_plan();
    pl->device = device;
    DeviceGuard guard(device);
    RomDev &D = pl->dev;
    D.n = n; D.E = E; D.n_bc = (int)bc_dof.size(); D.n_free = nf; D.hbw = hbw; D.bw1 = bw1; D.n_band = n_band;
    D.n_pairs = (int)pair_si.size();
    int rc = GPDE_OK;
    // the kernels' tables go into ONE arena (16-byte aligned pieces) that each CTA copies to shared memory
    std::vector<char> arena;
    auto put = [&arena](const void *src, size_t bytes) {
        const size_t off = (arena.size() + 15) & ~(size_t)15;
        arena.resize(off + bytes);
        if (bytes) memcpy(arena.data() + off, src, bytes);
        return off;
    };
#define AR(field, vec) const size_t off_##field = put(vec.data(), vec.size() * sizeof(vec[0]))
    AR(band_coef, band_coef); AR(rhs_coef, rhs_coef); AR(grad_coef, grad_coef); AR(cf_coef, cf_coef);
    AR(free_dof, free_dof); AR(bc_dof, bc_dof);
    AR(band_ptr, band_ptr); AR(band_elem, band_elem);
    AR(rhs_ptr, rhs_ptr); AR(rhs_elem, rhs_elem); AR(rhs_dof, rhs_dof);
    AR(grad_ptr, grad_ptr); AR(grad_i, grad_i); AR(grad_j, grad_j);
    AR(cf_ptr, cf_ptr); AR(cf_elem, cf_elem); AR(cf_free, cf_free);
    AR(pair_si, pair_si); AR(pair_sj, pair_sj);
#undef AR
    arena.resize((arena.size() + 15) & ~(size_t)15);
    const char *arena_dev = nullptr;
    if (rc == GPDE_OK) rc = track(pl, &arena_dev, arena);
    D.arena = arena_dev;
    D.arena_bytes = (int)arena.size();
#define SET(field) D.field = reinterpret_cast<decltype(D.field)>(arena_dev + off_##field)
    SET(band_coef); SET(rhs_coef); SET(grad_coef); SET(cf_coef); SET(free_dof); SET(bc_dof);
    SET(band_ptr); SET(band_elem); SET(rhs_ptr); SET(rhs_elem); SET(rhs_dof);
    SET(grad_ptr); SET(grad_i); SET(grad_j); SET(cf_ptr); SET(cf_elem); SET(cf_free); SET(pair_si); SET(pair_sj);
#undef SET
#define UP(field, vec) if (rc == GPDE_OK) rc = track(pl, &D.field, vec)
    UP(st_ptr, st_ptr); UP(st_elem, st_elem); UP(st_coef, st_coef); UP(is_bc, is_bc);
#undef UP
    if (rc != GPDE_OK) {
        gpde_rom_plan_destroy(pl);
        return rc;
    }
    const int pairs = D.n_pairs;
    pl->lanes = pairs <= 8 ? 8 : (pairs <= 16 ? 16 : 32);
    pl->n_contrib = (int)band_elem.size();
    // thread-per-sample kernels (rom_tps.cuh) when M fits their compile-time shape (the reference's 4x4 coarse mesh);
    // GPDE_ROM_PATH=coop keeps the plan on the cooperative kernels (A/B runs; read once, here).  Decided once per plan:
    // it fixes whether a factor stash exists.
    {
        const char *e = getenv("GPDE_ROM_PATH");
        const bool want = !(e && strcmp(e, "coop") == 0);
        pl->tps = (want && build_tps_tables<TpsShape4x4>(n, E, nf, hbw, free_dof, bc_dof, is_bc, M, pl->tps_tab)) ? 1 : 0;
        pl->tpw = 0;
        pl->tpw_fwd = nullptr;
        pl->tpw_adj = nullptr;
        if (want && !pl->tps) {
            std::vector<TpwFwdTab<TpwShape8x8>> ft(1);
            std::vector<TpwAdjTab<TpwShape8x8>> at(1);
            if (build_tpw_tables<TpwShape8x8>(n, E, nf, hbw, free_dof, bc_dof, is_bc, M, ft[0], at[0])) {
                int rc2 = track(pl, &pl->tpw_fwd, ft);
                if (rc2 == GPDE_OK) rc2 = track(pl, &pl->tpw_adj, at);
                if (rc2 != GPDE_OK) {
                    gpde_rom_plan_destroy(pl);
                    return rc2;
                }
                pl->tpw = 1;
            }
        }
    }
    // per-sample scratch of the cooperative kernels; with 8 lanes per sample a 64-bit shared-memory wavefront serves two
    // samples, so the pitch is padded to 8 (mod 16) doubles: the two samples' unit-stride accesses then fall on disjoint
    // halves of the banks
    auto pad_pitch = [&](size_t doubles) {
        if (pl->lanes != 8) return doubles;
        while (doubles % 16 != 8) ++doubles;
        return doubles;
    };
    pl->smem_fwd = sizeof(double) * pad_pitch((size_t)(E + n + n_band + 3 * nf));
    pl->smem_adj = sizeof(double) * pad_pitch((size_t)(2 * E + 2 * n + n_band + 4 * nf));
    const size_t groups = (kRomThreads / 32) * (32 / pl->lanes);
    if (groups * pl->smem_adj + arena.size() > 227 * 1024) {
        gpde_rom_plan_destroy(pl);
        return fail(GPDE_ERR_SIZE, "rom_plan_create: %zu bytes of shared memory per CTA exceed 227 KB",
                    groups * pl->smem_adj + arena.size());
    }
    *plan = pl;
    return GPDE_OK;
}

int gpde_rom_plan_destroy(gpde_rom_plan *pl) {
    if (!pl) return GPDE_OK;
    DeviceGuard guard(pl->device);
    for (void *p : pl->allocs) cudaFree(p);
    delete pl;
    return GPDE_OK;
}

int gpde_rom_plan_info(const gpde_rom_plan *pl, int64_t out[8]) {
    if (!pl || !out) return fail(GPDE_ERR_ARG, "rom_plan_info: null");
    out[0] = pl->dev.n; out[1] = pl->dev.E; out[2] = pl->dev.n_free; out[3] = pl->dev.hbw;
    // [4] doubles of factor stash per sample (0: none; windowed kernels: per sample of a 128-sample block -- size the buffer
    // with gpde_rom_factor_bytes); [6] lanes per sample: 1 = thread per sample (no stash), 2 = windowed thread per sample
    // (the forward call itself needs the stash), 8/16/32 = cooperative kernels
    out[4] = pl->tps ? 0 : (pl->tpw ? TpwShape8x8::NF * TpwShape8x8::W : pl->dev.n_band);
    out[5] = pl->n_contrib; out[6] = pl->tps ? 1 : (pl->tpw ? 2 : pl->lanes); out[7] = pl->device;
    return GPDE_OK;
}

size_t gpde_rom_factor_bytes(const gpde_rom_plan *pl, int64_t B) {
    if (!pl || B < 0 || pl->tps) return 0;   // the thread-per-sample kernels keep no stash
    if (pl->tpw)                              // sample-interleaved blocks of 128 samples
        return sizeof(double) * tpw_stash_doubles_per_block<TpwShape8x8>() * (size_t)((B + kTpwThreads - 1) / kTpwThreads);
    return sizeof(double) * (size_t)pl->dev.n_band * (size_t)B;
}

int gpde_rom_forward_f64(const gpde_rom_plan *pl, const double *X, int x_is_log, const double *F, double *u,
                         double *factor, int *info, int64_t B, gpde_stream_t stream) {
    return rom_forward<double>(pl, X, x_is_log, F, u, factor, info, B, stream);
}
int gpde_rom_forward_f32(const gpde_rom_plan *pl, const float *X, int x_is_log, const float *F, float *u,
                         double *factor, int *info, int64_t B, gpde_stream_t stream) {
    return rom_forward<float>(pl, X, x_is_log, F, u, factor, info, B, stream);
}
int gpde_rom_adjoint_f64(const gpde_rom_plan *pl, const double *X, int x_is_log, const double *u,
                         const double *factor, const double *gbar, double *gradX, double *gradF, int64_t B,
                         gpde_stream_t stream) {
    return rom_adjoint<double>(pl, X, x_is_log, u, factor, gbar, gradX, gradF, B, stream);
}
int gpde_rom_adjoint_f32(const gpde_rom_plan *pl, const float *X, int x_is_log, const float *u,
                         const double *factor, const float *gbar, float *gradX, float *gradF, int64_t B,
                         gpde_stream_t stream) {
    return rom_adjoint<float>(pl, X, x_is_log, u, factor, gbar, gradX, gradF, B, stream);
}

int gpde_rom_stiffness_f64(const gpde_rom_plan *pl, const double *X, double *K, int dirichlet, int64_t B,
                           gpde_stream_t stream) {
    if (!pl || B < 0) return fail(GPDE_ERR_ARG, "rom_stiffness: null plan or negative batch");
    if (B == 0) return GPDE_OK;
    if (!X || !K) return fail(GPDE_ERR_ARG, "rom_stiffness: null argument");
    DeviceGuard guard(pl->device);
    const long long total = (long long)pl->dev.n * pl->dev.n * B;
    const int threads = 256;
    const long long want = (total + threads - 1) / threads;
    const unsigned grid = (unsigned)std::min<long long>(want, (long long)sm_count(pl->device) * 16);
    rom_stiffness_kernel<<<grid, threads, 0, (cudaStream_t)stream>>>(pl->dev, X, K, dirichlet, B);
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

}  // extern "C"

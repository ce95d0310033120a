// Batched Gaussian conditioning of the virtual observables for 64 < m <= 256, matrix-free (sm_100a).  Included by vo.cu.
//
// Same algebra as vo_posterior.cuh (see its header comment); there Lambda and Lambda^-1 (m x m) live in shared memory,
// which caps m at 64.  Here the m x m matrices go to a caller-provided workspace in global memory (512 kB per data point
// for each of L and L^-1 at m = 256: they stay in L2) and the work is split over three launches.  m is padded to mp, a
// multiple of 64, and Lambda is handled as NB x NB blocks of 64 x 64 (NB = mp / 64; nbt = NB (NB + 1) / 2 lower blocks).
//
//   gram    grid (nbt * S, N): CTA (block (bi, bj), row segment s, data point n) streams its rows in tiles of 32, forms
//           K_ij(a) (post_tile_values), recomputes the two 64-column panels of q_r = (Gamma^T)_r it needs into shared
//           memory and accumulates  Lambda_blk += sum_r c_r q_r[bi] q_r[bj]^T  with mma.sync.m8n8k4.f64 (DMMA);
//           diagonal blocks also accumulate resid[bi] = V[:, bi]^T rho.  Gamma is never stored.  The CTAs of one data
//           point have adjacent numbers, so its V panels are read from L2 by all its blocks.  S > 1 (few data points)
//           splits the rows; every (segment, block) writes its partial block to the workspace.
//   factor  one CTA per data point: sums the S partials in segment order, adds diag(sigma^2) (identity on the padding),
//           then a blocked right-looking Cholesky in the workspace with 64 x 64 tiles staged through shared memory, the
//           explicit lower-triangular X = L^-1 and sol = Lambda^-1 resid = X^T (X resid).
//   apply   grid (tile of 32 rows, N): recomputes q_r for all mp columns, z_r = X q_r by DMMA with X streamed from L2
//           (only the lower triangle), vars_r = c_r - c_r^2 |z_r|^2 and mean_r = g_r - c_r q_r . sol.
// No atomics on results: every sum runs in a fixed order, so results are deterministic (for a given S: S depends on
// N, the SM count and d only).  gpde_vo_moments_f64 with m > 64 runs vo_moments_panel_kernel on (64-column panel, n).
#pragma once

namespace gpde {

constexpr int kBlkTile = 64;                 // side of a Lambda block
constexpr int kBlkRows = 32;                 // rows of a streamed tile (= kPostRows: one row per 8 threads)
constexpr int kBlkPitch = kBlkTile + 4;      // doubles per row of a 64-column q panel in shared memory (4 mod 16)
constexpr int kBlkTP = kBlkTile + 1;         // pitch of the factor kernel's 64 x 64 tiles

// q_r[c0 + cg + 8 j] (j < 8) for the thread's tile row r = tid / 8, cg = tid % 8; zero past column m / past the tile
__device__ __forceinline__ void blk_tile_panel(const VoCsrDev &C, const double *__restrict__ V, int m, int c0, int row0,
                                               int rows, const double *vals_s, double (&q)[8]) {
    const int r = threadIdx.x >> 3, cg = threadIdx.x & 7;
#pragma unroll
    for (int j = 0; j < 8; ++j) q[j] = 0.0;
    if (r < rows) {
        const int kbase = C.row_ptr[row0];
        const int k1 = C.row_ptr[row0 + r + 1];
        for (int k = C.row_ptr[row0 + r]; k < k1; ++k) {
            const double v = vals_s[k - kbase];
            const double *vr = V + (long long)C.col[k] * m + c0 + cg;
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (c0 + cg + 8 * j < m) q[j] = fma(v, __ldg(vr + 8 * j), q[j]);
        }
    }
}

// lower block number -> (bi, bj), bi >= bj, numbered row by row
__device__ __forceinline__ void blk_coords(int blk, int &bi, int &bj) {
    bi = 0;
    while ((bi + 1) * (bi + 2) / 2 <= blk) ++bi;
    bj = blk - bi * (bi + 1) / 2;
}

// Workspace of one data point (doubles): [0, pa) the S partials of the gram pass (segment s: nbt blocks of 64 x 64,
// then mp resid entries), later reused for X = L^-1 [mp][mp]; [pa, pa + mp^2) L; then sol [mp].
struct BlkLayout {
    int mp, nb, nbt, S;
    long long seg, pa, stride;    // doubles per partial segment, offset of L, doubles per data point
};

// ---- pass 1: Gram blocks and resid, partial over a row segment
// shared memory (doubles): Qa [32][68] | Qb [32][68] | vals [32 * max_row]
__global__ void __launch_bounds__(kPostThreads)
vo_post_gram_kernel(VoCsrDev C, const double *__restrict__ a, long long a_stride, const double *__restrict__ V,
                    long long v_stride, int m, const double *__restrict__ rho, const double *__restrict__ prec,
                    double *__restrict__ ws, BlkLayout Lo) {
    extern __shared__ __align__(16) double blk_smem[];
    double *Qa = blk_smem, *Qb = Qa + kBlkRows * kBlkPitch, *vals_s = Qb + kBlkRows * kBlkPitch;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r = tid >> 3, cg = tid & 7;
    const int blk = blockIdx.x / Lo.S, seg = blockIdx.x - blk * Lo.S;
    const long long n = blockIdx.y;
    int bi, bj;
    blk_coords(blk, bi, bj);
    const bool diag = bi == bj;
    const int d = C.d;
    const double *an = a + n * a_stride, *Vn = V + n * v_stride, *pn = prec + n * d, *rn = rho + n * d;
    const int tiles = (d + kBlkRows - 1) / kBlkRows;
    const int t0 = (int)((long long)tiles * seg / Lo.S), t1 = (int)((long long)tiles * (seg + 1) / Lo.S);
    const int wm = warp & 3, wn = warp >> 2;      // warp tile: rows 16 wm + [0, 16), columns 32 wn + [0, 32) of the block

    double acc[2][4][2];
#pragma unroll
    for (int x = 0; x < 2; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y][0] = acc[x][y][1] = 0.0;
    double rp[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) rp[j] = 0.0;

    for (int t = t0; t < t1; ++t) {
        const int row0 = t * kBlkRows, rows = min(kBlkRows, d - row0);
        __syncthreads();
        post_tile_values(C, an, row0, rows, vals_s);
        __syncthreads();
        double q[8];
        blk_tile_panel(C, Vn, m, kBlkTile * bj, row0, rows, vals_s, q);
        const double cr = r < rows ? 1.0 / pn[row0 + r] : 0.0;
#pragma unroll
        for (int j = 0; j < 8; ++j) Qb[r * kBlkPitch + cg + 8 * j] = q[j];
        if (diag) {
#pragma unroll
            for (int j = 0; j < 8; ++j) Qa[r * kBlkPitch + cg + 8 * j] = cr * q[j];
            if (r < rows) {
                const double rr = rn[row0 + r];
                const double *vr = Vn + (long long)(row0 + r) * m + kBlkTile * bi + cg;
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (kBlkTile * bi + cg + 8 * j < m) rp[j] = fma(__ldg(vr + 8 * j), rr, rp[j]);
            }
        } else {
            blk_tile_panel(C, Vn, m, kBlkTile * bi, row0, rows, vals_s, q);
#pragma unroll
            for (int j = 0; j < 8; ++j) Qa[r * kBlkPitch + cg + 8 * j] = cr * q[j];
        }
        __syncthreads();
        // block[i][j] += sum_r Qa[r][i] Qb[r][j]: A = Qa^T (8 x 4, row), B = Qb (4 x 8, col), k = the tile's rows
        const double *qa = Qa + (lane & 3) * kBlkPitch + 16 * wm + (lane >> 2);
        const double *qb = Qb + (lane & 3) * kBlkPitch + 32 * wn + (lane >> 2);
#pragma unroll
        for (int ks = 0; ks < kBlkRows / 4; ++ks) {
            double af[2], bf[4];
#pragma unroll
            for (int x = 0; x < 2; ++x) af[x] = qa[4 * ks * kBlkPitch + 8 * x];
#pragma unroll
            for (int y = 0; y < 4; ++y) bf[y] = qb[4 * ks * kBlkPitch + 8 * y];
#pragma unroll
            for (int x = 0; x < 2; ++x)
#pragma unroll
                for (int y = 0; y < 4; ++y) dmma884(acc[x][y][0], acc[x][y][1], af[x], bf[y]);
        }
    }
    double *part = ws + n * Lo.stride + seg * Lo.seg;
    double *pb = part + (long long)blk * kBlkTile * kBlkTile;
#pragma unroll
    for (int x = 0; x < 2; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            const int i = 16 * wm + 8 * x + (lane >> 2), j = 32 * wn + 8 * y + 2 * (lane & 3);
            *reinterpret_cast<double2 *>(pb + i * kBlkTile + j) = make_double2(acc[x][y][0], acc[x][y][1]);
        }
    if (diag) {     // resid[bi] over the segment: reduce the 32 row slots in order
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; ++j) Qa[r * kBlkPitch + cg + 8 * j] = rp[j];
        __syncthreads();
        if (tid < kBlkTile) {
            double s = 0.0;
            for (int rr = 0; rr < kBlkRows; ++rr) s += Qa[rr * kBlkPitch + tid];
            part[(long long)Lo.nbt * kBlkTile * kBlkTile + kBlkTile * bi + tid] = s;
        }
    }
}

// ---- factor kernel helpers (256 threads; thread t owns tile entries (t / 16 + 16 x, t % 16 + 16 y), x, y < 4)
__device__ __forceinline__ void blk_load_tile(double *dst, const double *src, int ld) {
    for (int e = threadIdx.x; e < kBlkTile * kBlkTile; e += kPostThreads) {
        const int i = e >> 6, j = e & 63;
        dst[i * kBlkTP + j] = src[(long long)i * ld + j];
    }
}
// acc[x][y] += sum_l A[i][l] B'[l][j], B' = B (transB = false) or B^T
template <bool TransB>
__device__ __forceinline__ void blk_tile_mma(double (&acc)[4][4], const double *A, const double *B) {
    const int ti = threadIdx.x >> 4, tj = threadIdx.x & 15;
    for (int l = 0; l < kBlkTile; ++l) {
        double av[4], bv[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) av[x] = A[(ti + 16 * x) * kBlkTP + l];
#pragma unroll
        for (int y = 0; y < 4; ++y) bv[y] = TransB ? B[(tj + 16 * y) * kBlkTP + l] : B[l * kBlkTP + tj + 16 * y];
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
            for (int y = 0; y < 4; ++y) acc[x][y] = fma(av[x], bv[y], acc[x][y]);
    }
}
__device__ __forceinline__ void blk_zero(double (&acc)[4][4]) {
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y] = 0.0;
}
// dst[i][j] = scale * acc (global, leading dimension ld) and, if sm != nullptr, the same into a shared tile
__device__ __forceinline__ void blk_store(const double (&acc)[4][4], double scale, double *dst, int ld, double *sm) {
    const int ti = threadIdx.x >> 4, tj = threadIdx.x & 15;
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            const int i = ti + 16 * x, j = tj + 16 * y;
            dst[(long long)i * ld + j] = scale * acc[x][y];
            if (sm) sm[i * kBlkTP + j] = scale * acc[x][y];
        }
}

// ---- pass 2: assemble Lambda, Cholesky, X = L^-1, sol
// shared memory (doubles): T0, T1, P[3] tiles of [64][65] | resid [mp] | z [mp]
__global__ void __launch_bounds__(kPostThreads)
vo_post_factor_kernel(int m, const double *__restrict__ noise_var, double *__restrict__ ws, BlkLayout Lo, int *info) {
    extern __shared__ __align__(16) double blk_smem[];
    constexpr int TS = kBlkTile * kBlkTP;
    double *T0 = blk_smem, *T1 = T0 + TS, *P = T1 + TS, *rs = P + 3 * TS, *zs = rs + Lo.mp;
    const int tid = threadIdx.x, mp = Lo.mp, NB = Lo.nb;
    const long long n = blockIdx.x;
    double *base = ws + n * Lo.stride;
    double *L = base + Lo.pa, *X = base, *sol = L + (long long)mp * mp;

    // Lambda (lower blocks) = sum of the partials in segment order + diag(sigma^2); resid likewise
    for (int blk = 0; blk < Lo.nbt; ++blk) {
        int bi, bj;
        blk_coords(blk, bi, bj);
        for (int e = tid; e < kBlkTile * kBlkTile; e += kPostThreads) {
            const int i = e >> 6, j = e & 63;
            double v = 0.0;
            for (int s = 0; s < Lo.S; ++s) v += base[s * Lo.seg + (long long)blk * kBlkTile * kBlkTile + e];
            if (bi == bj && i == j) v += kBlkTile * bi + i < m ? noise_var[kBlkTile * bi + i] : 1.0;   // padding: identity
            L[(long long)(kBlkTile * bi + i) * mp + kBlkTile * bj + j] = v;
        }
    }
    for (int c = tid; c < mp; c += kPostThreads) {
        double v = 0.0;
        for (int s = 0; s < Lo.S; ++s) v += base[s * Lo.seg + (long long)Lo.nbt * kBlkTile * kBlkTile + c];
        rs[c] = v;
    }
    __syncthreads();     // the partials are consumed: X may overwrite them from here on

    int bad = 0;
    double acc[4][4];
    for (int k = 0; k < NB; ++k) {
        double *Lkk = L + (long long)kBlkTile * k * mp + kBlkTile * k;
        blk_load_tile(T0, Lkk, mp);
        __syncthreads();
        // unblocked Cholesky of the diagonal tile: step j updates the trailing triangle from the unscaled column j, then
        // scales column j (the next step reads column j + 1 only, so one barrier per step suffices)
        for (int j = 0; j < kBlkTile; ++j) {
            const double piv = T0[j * kBlkTP + j];
            if (!(piv > 0.0)) bad = 1;
            const double rpiv = 1.0 / piv;
            for (int e = tid; e < kBlkTile * kBlkTile; e += kPostThreads) {
                const int i = e >> 6, l = e & 63;
                if (l > j && i >= l) T0[i * kBlkTP + l] -= T0[i * kBlkTP + j] * T0[l * kBlkTP + j] * rpiv;
            }
            __syncthreads();
            const double ljj = sqrt(piv);
            if (tid < kBlkTile && tid >= j) T0[tid * kBlkTP + j] = tid == j ? ljj : T0[tid * kBlkTP + j] / ljj;
        }
        __syncthreads();
        // T1 = T0^-1 (lower): column c by thread c, forward substitution
        if (tid < kBlkTile) {
            const int c = tid;
            for (int i = 0; i < kBlkTile; ++i) {
                double s = i == c ? 1.0 : 0.0;
                for (int l = c; l < i; ++l) s -= T0[i * kBlkTP + l] * T1[l * kBlkTP + c];
                T1[i * kBlkTP + c] = i < c ? 0.0 : s / T0[i * kBlkTP + i];
            }
        }
        __syncthreads();
        for (int e = tid; e < kBlkTile * kBlkTile; e += kPostThreads) {
            const int i = e >> 6, j = e & 63;
            Lkk[(long long)i * mp + j] = j <= i ? T0[i * kBlkTP + j] : 0.0;
            X[(long long)(kBlkTile * k + i) * mp + kBlkTile * k + j] = T1[i * kBlkTP + j];    // X_kk = L_kk^-1
        }
        // panel: L_ik = A_ik L_kk^-T, kept in P[i - k - 1] for the trailing update
        for (int i = k + 1; i < NB; ++i) {
            double *Pi = P + (i - k - 1) * TS;
            blk_load_tile(Pi, L + (long long)kBlkTile * i * mp + kBlkTile * k, mp);
            __syncthreads();
            blk_zero(acc);
            blk_tile_mma<true>(acc, Pi, T1);
            __syncthreads();
            blk_store(acc, 1.0, L + (long long)kBlkTile * i * mp + kBlkTile * k, mp, Pi);
        }
        __syncthreads();
        // trailing update A_ij -= L_ik L_jk^T  (k < j <= i)
        for (int j = k + 1; j < NB; ++j)
            for (int i = j; i < NB; ++i) {
                double *Aij = L + (long long)kBlkTile * i * mp + kBlkTile * j;
                const int ti = tid >> 4, tj = tid & 15;
#pragma unroll
                for (int x = 0; x < 4; ++x)
#pragma unroll
                    for (int y = 0; y < 4; ++y) acc[x][y] = Aij[(long long)(ti + 16 * x) * mp + tj + 16 * y];
                double neg[4][4];
                blk_zero(neg);
                blk_tile_mma<true>(neg, P + (i - k - 1) * TS, P + (j - k - 1) * TS);
#pragma unroll
                for (int x = 0; x < 4; ++x)
#pragma unroll
                    for (int y = 0; y < 4; ++y) acc[x][y] -= neg[x][y];
                blk_store(acc, 1.0, Aij, mp, nullptr);
            }
        __syncthreads();
    }
    if (bad && tid == 0 && info) atomicOr(info, GPDE_INFO_NOT_SPD);

    // X_ij = -X_ii sum_{l = j}^{i - 1} L_il X_lj  (i > j), block column by block column, top to bottom
    for (int j = 0; j < NB; ++j)
        for (int i = j + 1; i < NB; ++i) {
            blk_zero(acc);
            for (int l = j; l < i; ++l) {
                blk_load_tile(T0, L + (long long)kBlkTile * i * mp + kBlkTile * l, mp);
                blk_load_tile(T1, X + (long long)kBlkTile * l * mp + kBlkTile * j, mp);
                __syncthreads();
                blk_tile_mma<false>(acc, T0, T1);
                __syncthreads();
            }
            blk_store(acc, 1.0, X + (long long)kBlkTile * i * mp + kBlkTile * j, mp, P);     // P = S_ij
            blk_load_tile(T0, X + (long long)kBlkTile * i * mp + kBlkTile * i, mp);
            __syncthreads();
            blk_zero(acc);
            blk_tile_mma<false>(acc, T0, P);
            __syncthreads();
            blk_store(acc, -1.0, X + (long long)kBlkTile * i * mp + kBlkTile * j, mp, nullptr);
            __syncthreads();
        }
    __syncthreads();
    // sol = X^T (X resid): z_i = sum_{k <= i} X_ik resid_k, sol_k = sum_{i >= k} X_ik z_i
    for (int i = tid; i < mp; i += kPostThreads) {
        double s = 0.0;
        for (int k = 0; k <= i; ++k) s = fma(X[(long long)i * mp + k], rs[k], s);
        zs[i] = s;
    }
    __syncthreads();
    for (int k = tid; k < mp; k += kPostThreads) {
        double s = 0.0;
        for (int i = k; i < mp; ++i) s = fma(X[(long long)i * mp + k], zs[i], s);
        sol[k] = k < m ? s : 0.0;
    }
}

// ---- pass 3: mean and vars of a tile of 32 rows
// shared memory (doubles): Q [32][mp + 4] | vals [32 * max_row] | sol [mp] | quad partials [8 warps][32] | lin [32]
__global__ void __launch_bounds__(kPostThreads)
vo_post_apply_kernel(VoCsrDev C, const double *__restrict__ a, long long a_stride, const double *__restrict__ V,
                     long long v_stride, int m, const double *__restrict__ g, const double *__restrict__ prec,
                     const double *__restrict__ ws, BlkLayout Lo, double *__restrict__ mean, double *__restrict__ vars) {
    extern __shared__ __align__(16) double blk_smem[];
    const int mp = Lo.mp, QP = mp + 4;
    double *Q = blk_smem, *vals_s = Q + kBlkRows * QP, *sol_s = vals_s + kBlkRows * C.max_row;
    double *red = sol_s + mp, *lin_s = red + 8 * kBlkRows;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, r = tid >> 3, cg = tid & 7;
    const long long n = blockIdx.y;
    const int d = C.d, row0 = blockIdx.x * kBlkRows, rows = min(kBlkRows, d - row0);
    const double *an = a + n * a_stride, *Vn = V + n * v_stride;
    const double *X = ws + n * Lo.stride, *sol = X + Lo.pa + (long long)mp * mp;
    for (int c = tid; c < mp; c += kPostThreads) sol_s[c] = sol[c];
    post_tile_values(C, an, row0, rows, vals_s);
    __syncthreads();
    double lin = 0.0;
    for (int p = 0; p < Lo.nb; ++p) {
        double q[8];
        blk_tile_panel(C, Vn, m, kBlkTile * p, row0, rows, vals_s, q);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            Q[r * QP + kBlkTile * p + cg + 8 * j] = q[j];
            lin = fma(q[j], sol_s[kBlkTile * p + cg + 8 * j], lin);
        }
    }
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) lin += __shfl_xor_sync(0xffffffffu, lin, o);
    if (cg == 0) lin_s[r] = lin;
    __syncthreads();
    // |X q_r|^2: D[r][i] = sum_k Q[r][k] X[i][k] over k < 8 (nt + 1) (X lower triangular), A = Q (row), B = X^T (col).
    // 8-column tiles nt and NT - 1 - nt go to the same warp: every warp gets the same number of k-steps.
    const int NT = mp / 8;
    double ss[4] = {0.0, 0.0, 0.0, 0.0};
    const double *qa = Q + (lane >> 2) * QP + (lane & 3);
    for (int nt = 0; nt < NT; ++nt) {
        if (((nt < NT / 2 ? nt : NT - 1 - nt) & 7) != warp) continue;
        const double *xb = X + (long long)(8 * nt + (lane >> 2)) * mp + (lane & 3);
        double acc[4][2];
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) acc[mt][0] = acc[mt][1] = 0.0;
        const int ksteps = 2 * nt + 2;
#pragma unroll 4
        for (int ks = 0; ks < ksteps; ++ks) {
            const double bf = __ldg(xb + 4 * ks);
#pragma unroll
            for (int mt = 0; mt < 4; ++mt) dmma884(acc[mt][0], acc[mt][1], qa[8 * mt * QP + 4 * ks], bf);
        }
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) ss[mt] = fma(acc[mt][0], acc[mt][0], fma(acc[mt][1], acc[mt][1], ss[mt]));
    }
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) {
        ss[mt] += __shfl_xor_sync(0xffffffffu, ss[mt], 1);
        ss[mt] += __shfl_xor_sync(0xffffffffu, ss[mt], 2);
        if ((lane & 3) == 0) red[warp * kBlkRows + 8 * mt + (lane >> 2)] = ss[mt];
    }
    __syncthreads();
    if (tid < rows) {
        double quad = 0.0;
        for (int w = 0; w < 8; ++w) quad += red[w * kBlkRows + tid];
        const long long o = n * d + row0 + tid;
        const double cr = 1.0 / prec[o];
        mean[o] = g[o] - cr * lin_s[tid];
        vars[o] = cr - cr * cr * quad;
    }
}

// ---- moments for m > 64: vo_moments_kernel's per-column logic on the 64-column panel blockIdx.x of data point blockIdx.y
__global__ void __launch_bounds__(kPostThreads, 1)
vo_moments_panel_kernel(VoCsrDev C, const double *__restrict__ a, long long a_stride, const double *__restrict__ V,
                        long long v_stride, int m, const double *__restrict__ rho, const double *__restrict__ v,
                        double *__restrict__ out_r, double *__restrict__ out_s2) {
    extern __shared__ __align__(16) double post_smem[];
    double *vals_s = post_smem;
    double *red = vals_s + kPostRows * C.max_row;      // [2][32][64]
    const int tid = threadIdx.x, r = tid >> 3, cg = tid & 7;
    const int c0 = kBlkTile * blockIdx.x;
    const long long n = blockIdx.y;
    const double *an = a + n * a_stride, *Vn = V + n * v_stride, *vn = v + n * C.d, *rn = rho + n * C.d;
    double part[8], rp[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) part[j] = rp[j] = 0.0;
    for (int row0 = 0; row0 < C.d; row0 += kPostRows) {
        const int rows = min(kPostRows, C.d - row0);
        __syncthreads();
        post_tile_values(C, an, row0, rows, vals_s);
        __syncthreads();
        double q[8];
        blk_tile_panel(C, Vn, m, c0, row0, rows, vals_s, q);
        if (r < rows) {
            const double w = vn[row0 + r], rr = rn[row0 + r];
            const double *vr = Vn + (long long)(row0 + r) * m + c0 + cg;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                part[j] = fma(q[j] * q[j], w, part[j]);
                if (c0 + cg + 8 * j < m) rp[j] = fma(__ldg(vr + 8 * j), rr, rp[j]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        red[r * kBlkTile + cg + 8 * j] = part[j];
        red[(kPostRows + r) * kBlkTile + cg + 8 * j] = rp[j];
    }
    __syncthreads();
    const int mc = min(kBlkTile, m - c0);
    for (int c = tid; c < 2 * mc; c += kPostThreads) {
        const int which = c >= mc, cc = c - which * mc;
        double s = 0.0;
        for (int rr = 0; rr < kPostRows; ++rr) s += red[(which * kPostRows + rr) * kBlkTile + cc];
        (which ? out_r : out_s2)[n * m + c0 + cc] = s;
    }
}

static inline size_t blk_gram_smem(int max_row) {
    return sizeof(double) * ((size_t)2 * kBlkRows * kBlkPitch + (size_t)kBlkRows * max_row);
}
static inline size_t blk_factor_smem(int mp) {
    return sizeof(double) * ((size_t)5 * kBlkTile * kBlkTP + (size_t)2 * mp);
}
static inline size_t blk_apply_smem(int mp, int max_row) {
    return sizeof(double) * ((size_t)kBlkRows * (mp + 4) + (size_t)kBlkRows * max_row + mp + 9 * kBlkRows);
}
static inline size_t blk_moments_smem(int max_row) {
    return sizeof(double) * ((size_t)kPostRows * max_row + (size_t)2 * kPostRows * kBlkTile);
}

}  // namespace gpde

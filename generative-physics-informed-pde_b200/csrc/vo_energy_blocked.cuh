// Batched subspace-Newton step of the energy-type virtual observables for 64 < m <= 256, matrix-free (sm_100a).  Included
// by vo.cu after vo_posterior_blocked.cuh, whose layout, tile helpers and factor kernel it reuses (vo_post_gram_kernel
// itself is left as it is: this gram pass differs in its operands, so it has its own body).
//
// Same algebra as vo_energy.cuh (see its header comment); there M (m x m) lives in shared memory, which caps m at 64.
// Per data point n (inv_T = 1/T_n), with rho = K_ff(a) mean - f_eff from one rho-only residual launch before this step:
//   M    = sum_r V_r^T w_r,      w_r = prec_r V_r + inv_T q_r,   q_r = (K_ff(a) V)_r
//   b    = sum_r V_r grad_r,     grad_r = prec_r (mean_r - g_r) + inv_T rho_r
//   mean <- mean - V M^-1 b
// m is padded to mp (a multiple of 64) and M is handled as 64 x 64 lower blocks in the workspace of the blocked posterior
// (BlkLayout, blocked_layout in vo.cu: the same layout and size).  Three launches:
//   gram    grid (nbt * S, N), as vo_post_gram_kernel: CTA (block (bi, bj), row segment s, data point n) streams its rows
//           in tiles of 32, stages the plain V panel bi and the w panel bj (one q panel from post_tile_values /
//           blk_tile_panel) in shared memory and accumulates  M_blk += sum_r V_r[bi] w_r[bj]^T  by DMMA; diagonal blocks
//           also accumulate b[bi] into the slot of the posterior's resid.  Partial blocks go to the workspace, no atomics.
//   factor  vo_post_factor_kernel unchanged, with zero noise variances: sums the partials in segment order, identity on
//           the padding, Cholesky, X = L^-1 and sol = M^-1 b.  A non-positive pivot ORs GPDE_INFO_NOT_SPD into info.
//   apply   grid (tile of kEnergyApplyRows rows, N): mean_r -= V_r . sol on the rows of V alone (no CSR), one warp per row
//           with a fixed sum order.  A data point whose L has a diagonal entry that is not > 0 (the factor kernel stores
//           sqrt(pivot) there: exactly its non-positive-pivot test) keeps its mean bitwise.
// Results are deterministic for a given (plan, N, m): S depends on N, the SM count and d only.
#pragma once

namespace gpde {

constexpr int kEnergyApplyRows = 128;        // rows of V per apply CTA (16 per warp)

// zero noise variances for vo_post_factor_kernel (Lambda + diag(0) = M)
__device__ double energy_zero_noise[4 * kBlkTile];

// ---- pass 1: Gram blocks of M and b, partial over a row segment
// shared memory (doubles): Vs [32][68] | Ws [32][68] | vals [32 * max_row]  (blk_gram_smem)
__global__ void __launch_bounds__(kPostThreads)
vo_energy_gram_kernel(VoCsrDev C, const double *__restrict__ a, long long a_stride, const double *__restrict__ V,
                      long long v_stride, int m, const double *__restrict__ rho, const double *__restrict__ g,
                      const double *__restrict__ prec, const double *__restrict__ inv_T, const double *__restrict__ mean,
                      double *__restrict__ ws, BlkLayout Lo) {
    extern __shared__ __align__(16) double blk_smem[];
    double *Vs = blk_smem, *Ws = Vs + kBlkRows * kBlkPitch, *vals_s = Ws + kBlkRows * kBlkPitch;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, r = tid >> 3, cg = tid & 7;
    const int blk = blockIdx.x / Lo.S, seg = blockIdx.x - blk * Lo.S;
    const long long n = blockIdx.y;
    int bi, bj;
    blk_coords(blk, bi, bj);
    const bool diag = bi == bj;
    const int d = C.d;
    const double *an = a + n * a_stride, *Vn = V + n * v_stride;
    const double *pn = prec + n * d, *rn = rho + n * d, *gn = g + n * d, *mn = mean + n * d;
    const double it = inv_T[n];
    const int tiles = (d + kBlkRows - 1) / kBlkRows;
    const int t0 = (int)((long long)tiles * seg / Lo.S), t1 = (int)((long long)tiles * (seg + 1) / Lo.S);
    const int wm = warp & 3, wn = warp >> 2;      // warp tile: rows 16 wm + [0, 16), columns 32 wn + [0, 32) of the block

    double acc[2][4][2];
#pragma unroll
    for (int x = 0; x < 2; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y][0] = acc[x][y][1] = 0.0;
    double bp[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) bp[j] = 0.0;

    for (int t = t0; t < t1; ++t) {
        const int row0 = t * kBlkRows, rows = min(kBlkRows, d - row0);
        __syncthreads();
        post_tile_values(C, an, row0, rows, vals_s);
        __syncthreads();
        double q[8];
        blk_tile_panel(C, Vn, m, kBlkTile * bj, row0, rows, vals_s, q);
        const bool live = r < rows;
        const double *vr = Vn + (long long)(row0 + r) * m;      // read only for live rows
        double pr = 0.0, gr = 0.0;
        if (live) {
            pr = pn[row0 + r];
            if (diag) gr = pr * (mn[row0 + r] - gn[row0 + r]) + it * rn[row0 + r];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int c = kBlkTile * bj + cg + 8 * j;
            const double v = live && c < m ? __ldg(vr + c) : 0.0;
            Ws[r * kBlkPitch + cg + 8 * j] = pr * v + it * q[j];
            if (diag) {
                Vs[r * kBlkPitch + cg + 8 * j] = v;
                bp[j] = fma(v, gr, bp[j]);
            }
        }
        if (!diag) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int c = kBlkTile * bi + cg + 8 * j;
                Vs[r * kBlkPitch + cg + 8 * j] = live && c < m ? __ldg(vr + c) : 0.0;
            }
        }
        __syncthreads();
        // block[i][j] += sum_r Vs[r][i] Ws[r][j]: the DMMA fragment loop of vo_post_gram_kernel (A = Vs^T, B = Ws)
        const double *qa = Vs + (lane & 3) * kBlkPitch + 16 * wm + (lane >> 2);
        const double *qb = Ws + (lane & 3) * kBlkPitch + 32 * wn + (lane >> 2);
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
    if (diag) {     // b[bi] over the segment, into the resid slot: reduce the 32 row slots in order
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 8; ++j) Vs[r * kBlkPitch + cg + 8 * j] = bp[j];
        __syncthreads();
        if (tid < kBlkTile) {
            double s = 0.0;
            for (int rr = 0; rr < kBlkRows; ++rr) s += Vs[rr * kBlkPitch + tid];
            part[(long long)Lo.nbt * kBlkTile * kBlkTile + kBlkTile * bi + tid] = s;
        }
    }
}

// ---- pass 3: mean_r -= V_r . sol for a tile of kEnergyApplyRows rows
__global__ void __launch_bounds__(kPostThreads)
vo_energy_apply_kernel(int d, const double *__restrict__ V, long long v_stride, int m, const double *__restrict__ ws,
                       BlkLayout Lo, double *__restrict__ mean) {
    __shared__ double sol_s[4 * kBlkTile];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long n = blockIdx.y;
    const int mp = Lo.mp;
    const double *L = ws + n * Lo.stride + Lo.pa, *sol = L + (long long)mp * mp;
    int bad = 0;
    if (tid < mp) {
        bad = !(L[(long long)tid * (mp + 1)] > 0.0);
        sol_s[tid] = sol[tid];
    }
    if (__syncthreads_or(bad)) return;
    const double *Vn = V + n * v_stride;
    double *mn = mean + n * d;
    const int row0 = blockIdx.x * kEnergyApplyRows;
    for (int rr = warp; rr < kEnergyApplyRows; rr += kPostThreads / 32) {
        const int i = row0 + rr;
        if (i >= d) break;
        const double *vr = Vn + (long long)i * m;
        double s = 0.0;
        for (int c = lane; c < m; c += 32) s = fma(__ldg(vr + c), sol_s[c], s);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) mn[i] -= s;
    }
}

}  // namespace gpde

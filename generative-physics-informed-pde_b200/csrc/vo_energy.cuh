// Batched subspace-Newton step of the energy-type virtual observables, matrix-free (sm_100a).  Included by vo.cu after
// vo_posterior.cuh, whose CSR term lists and tile helpers it reuses.
//
// Reference (per data point, dense A = diag(prec) + K/T on the CPU):
//   EnergyVirtualObservable.update     bottleneck/VirtualObservables.py:769-788, looped over the data points at :1001-1037
//       mean <- mean - V (V^T A V)^-1 V^T (A mean - b),   b = f/T + prec g
// Per data point n (inv_T = 1/T_n), with rho = K_ff(a) mean - f_eff from one rho-only residual launch before this one:
//   M   = V^T diag(prec) V + inv_T V^T K_ff(a) V  = sum_r V_r^T w_r,   w_r = prec_r V_r + inv_T q_r,  q_r = (K_ff(a) V)_r
//   b   = V^T (prec (mean - g) + inv_T rho)       = sum_r V_r grad_r
//   mean <- mean - V M^-1 b
// One CTA owns one data point and streams over tiles of 32 free rows:
//   pass A   q tile from the CSR term lists (post_tile_values / post_tile_rows), V and w tiles -> shared memory;
//            M += V_tile^T w_tile (register blocks of the m x m matrix, 256 threads), b partials per thread
//   middle   identity padding to MP; Cholesky and two triangular solves in shared memory (warp 0): sol = M^-1 b.
//            A non-positive pivot ORs GPDE_INFO_NOT_SPD into info and leaves this data point's mean as it was.
//   pass B   mean_r -= V_r . sol (rows of V only, no CSR)
// V is shared by the data points (v_stride = 0) or one matrix per data point (v_stride = d m).
#pragma once

namespace gpde {

// shared memory (doubles): M [MP][MP+1] | Vs [32][MP+2] | Ws [32][MP+2] | vals [32 * max_row] | b [MP]
template <int MP>
__global__ void __launch_bounds__(kPostThreads)
vo_energy_step_kernel(VoCsrDev C, const double *__restrict__ a, long long a_stride, const double *__restrict__ V,
                      long long v_stride, int m, const double *__restrict__ rho, const double *__restrict__ g,
                      const double *__restrict__ prec, const double *__restrict__ inv_T, double *mean, int *info) {
    extern __shared__ __align__(16) double energy_smem[];
    __shared__ int bad_s;
    constexpr int LP = MP + 1, QP = MP + 2, BS = MP / 16;
    double *Ms = energy_smem;
    double *Vs = Ms + MP * LP;
    double *Ws = Vs + kPostRows * QP;
    double *vals_s = Ws + kPostRows * QP;
    double *bs = vals_s + kPostRows * C.max_row;
    const int tid = threadIdx.x;
    const long long n = blockIdx.x;
    const int d = C.d;
    const double *an = a + n * a_stride, *Vn = V + n * v_stride;
    const double *gn = g + n * d, *pn = prec + n * d, *rn = rho + n * d;
    double *mn = mean + n * d;
    const double it = inv_T[n];
    const int r = tid >> 3, cg = tid & 7;
    const int bi = tid >> 4, bj = tid & 15;

    // ---- pass A: M = sum_r V_r^T w_r,  b = sum_r V_r grad_r
    double acc[BS][BS];
#pragma unroll
    for (int x = 0; x < BS; ++x)
#pragma unroll
        for (int y = 0; y < BS; ++y) acc[x][y] = 0.0;
    double bp[MP / 8];          // partial sums of b over the thread's rows
#pragma unroll
    for (int j = 0; j < MP / 8; ++j) bp[j] = 0.0;
    for (int row0 = 0; row0 < d; row0 += kPostRows) {
        const int rows = min(kPostRows, d - row0);
        __syncthreads();
        post_tile_values(C, an, row0, rows, vals_s);
        __syncthreads();
        double q[MP / 8];
        post_tile_rows<MP>(C, Vn, m, row0, rows, vals_s, q);
        double pr = 0.0, gr = 0.0;
        const double *vr = Vn;
        if (r < rows) {
            const int i = row0 + r;
            pr = pn[i];
            gr = pr * (mn[i] - gn[i]) + it * rn[i];
            vr = Vn + (long long)i * m + cg;
        }
#pragma unroll
        for (int j = 0; j < MP / 8; ++j) {
            const int c = cg + 8 * j;
            const double v = (r < rows && c < m) ? __ldg(vr + 8 * j) : 0.0;
            bp[j] = fma(v, gr, bp[j]);
            Vs[r * QP + c] = v;
            Ws[r * QP + c] = pr * v + it * q[j];
        }
        __syncthreads();
#pragma unroll 4
        for (int rr = 0; rr < kPostRows; ++rr) {
            double va[BS], wb[BS];
#pragma unroll
            for (int x = 0; x < BS; ++x) {
                va[x] = Vs[rr * QP + BS * bi + x];
                wb[x] = Ws[rr * QP + BS * bj + x];
            }
#pragma unroll
            for (int x = 0; x < BS; ++x)
#pragma unroll
                for (int y = 0; y < BS; ++y) acc[x][y] = fma(va[x], wb[y], acc[x][y]);
        }
    }
    __syncthreads();
#pragma unroll
    for (int x = 0; x < BS; ++x)
#pragma unroll
        for (int y = 0; y < BS; ++y) {
            const int i = BS * bi + x, j = BS * bj + y;
            Ms[i * LP + j] = (i == j && i >= m) ? 1.0 : acc[x][y];      // padding rows / columns: identity
        }
#pragma unroll
    for (int j = 0; j < MP / 8; ++j) Vs[r * QP + cg + 8 * j] = bp[j];     // Vs is free: reduce b over the 32 row slots
    __syncthreads();
    for (int c = tid; c < MP; c += kPostThreads) {
        double sum = 0.0;
        for (int rr = 0; rr < kPostRows; ++rr) sum += Vs[rr * QP + c];
        bs[c] = sum;
    }
    __syncthreads();

    // ---- Cholesky M = L L^T (lower, in place), then L y = b and L^T sol = y in place on bs: warp 0, m <= 64
    if (tid < 32) {
        const int lane = tid;
        int bad = 0;
        for (int k = 0; k < MP; ++k) {
            const double dkk = Ms[k * LP + k];
            if (!(dkk > 0.0)) bad = 1;
            const double lkk = sqrt(dkk);
            __syncwarp();
            for (int i = k + lane; i < MP; i += 32) Ms[i * LP + k] = (i == k) ? lkk : Ms[i * LP + k] / lkk;
            __syncwarp();
            for (int j = k + 1 + lane; j < MP; j += 32) {       // column j of the trailing block (rows >= j)
                const double ljk = Ms[j * LP + k];
                for (int i = j; i < MP; ++i) Ms[i * LP + j] -= Ms[i * LP + k] * ljk;
            }
            __syncwarp();
        }
        for (int k = 0; k < MP; ++k) {                          // forward: y_k, then b_i -= L_ik y_k below it
            const double yk = bs[k] / Ms[k * LP + k];
            __syncwarp();
            if (lane == 0) bs[k] = yk;
            for (int i = k + 1 + lane; i < MP; i += 32) bs[i] -= Ms[i * LP + k] * yk;
            __syncwarp();
        }
        for (int k = MP - 1; k >= 0; --k) {                     // backward: sol_k, then y_i -= L_ki sol_k above it
            const double sk = bs[k] / Ms[k * LP + k];
            __syncwarp();
            if (lane == 0) bs[k] = sk;
            for (int i = lane; i < k; i += 32) bs[i] -= Ms[k * LP + i] * sk;
            __syncwarp();
        }
        if (lane == 0) {
            bad_s = bad;
            if (bad && info) atomicOr(info, GPDE_INFO_NOT_SPD);
        }
    }
    __syncthreads();
    if (bad_s) return;

    // ---- pass B: mean_r -= V_r . sol, 8 threads per row
    for (int row0 = 0; row0 < d; row0 += kPostRows) {
        const int i = row0 + r;
        double s = 0.0;
        if (i < d) {
            const double *vr = Vn + (long long)i * m;
#pragma unroll
            for (int j = 0; j < MP / 8; ++j) {
                const int c = cg + 8 * j;
                if (c < m) s = fma(__ldg(vr + c), bs[c], s);
            }
        }
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (cg == 0 && i < d) mn[i] -= s;
    }
}

template <int MP>
static inline size_t energy_smem_bytes(int max_row) {
    return sizeof(double) * ((size_t)MP * (MP + 1) + 2 * kPostRows * (MP + 2) + (size_t)kPostRows * max_row + MP);
}

}  // namespace gpde

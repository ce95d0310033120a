// One weighting matrix per sample: V [B,d,m] (V_b = V + b d m).  Included by vo.cu.
//
// The residual family with a per-sample V (gpde_vo_residual_*, _T_*, _grad_* with v_stride = d*m) reuses the shared-V
// routes' launches for everything that involves K(a): the rho-only residual, the K_ff application of residual_T and the
// gradient kernels of vo_grad.cuh.  What changes with a per-sample V is the contraction with V, which these kernels do:
//   vo_vb_contract_kernel   r[b,:] = V_b^T rho_b
//   vo_vb_expand_kernel     w[b,:] = V_b s_b          (FP64 rows of pitch ldw, the input of the K_ff application)
// Both stream V_b once (8 d m bytes per sample in FP64, against 8 d for rho_b or w_b): they are bound by HBM bandwidth,
// and there is no reuse of V across samples for a tensor-core tile to exploit.  FP32 I/O reads V, rho and s as floats
// and accumulates in FP64.  Every output is summed in a fixed order that does not depend on the grid: results are
// bitwise reproducible.
//
// The moments kernel (vo_posterior.cuh) also forms V_n^T rho_n, but inside its loop over the CSR row tiles, with the
// row-to-thread mapping and the reduction buffer it shares with s2 (8 lanes per row, at most 64 columns in registers).
// A device function common to both would impose that mapping on the streaming kernel here, so the two stay separate.
#pragma once

namespace gpde {

constexpr int kVbThreads = 256;   // contraction CTA
constexpr int kVbPanel = 64;      // columns of V per panel (any m: ceil(m / 64) panels)
constexpr int kVbRows = 64;       // rows of V_b per expansion tile
constexpr int kVbExpThreads = 128;   // expansion CTA: two threads per row
constexpr int kVbPitch = 66;      // doubles per staged row (interleaved halves: conflict-free, see vo_vb_expand_kernel)

// r[b, c0 + c] = sum_i V_b[i, c0 + c] rho_b[i] for the panel of P = min(64, m - c0) columns at c0; one CTA iteration per
// (sample, panel).  The P columns are spread over R = 256 / P row slots: thread t takes column t % P and the rows
// t / P, t / P + R, ...  For m <= 64 a pass of the CTA reads R whole consecutive rows, R m contiguous elements.  A thread
// adds its rows in ascending order; the R slot sums of a column are then added in slot order.
template <typename T>
__global__ void __launch_bounds__(kVbThreads)
vo_vb_contract_kernel(const T *__restrict__ V, const T *__restrict__ rho, T *__restrict__ r, int d, int m, long long B) {
    __shared__ double part[kVbThreads];
    const int npan = (m + kVbPanel - 1) / kVbPanel;
    const int t = threadIdx.x;
    for (long long job = blockIdx.x; job < B * npan; job += gridDim.x) {
        const long long b = job / npan;
        const int c0 = (int)(job - b * npan) * kVbPanel;
        const int P = min(kVbPanel, m - c0), R = kVbThreads / P;
        const int slot = t / P, c = t - slot * P;
        double acc = 0.0;
        if (slot < R) {
            const T *Vb = V + b * (long long)d * m + c0 + c;
            const T *rb = rho + b * d;
            int i = slot;
            for (; i + 3 * R < d; i += 4 * R) {   // four independent loads of V in flight per thread
                const double v0 = ldd(Vb + (long long)i * m), v1 = ldd(Vb + (long long)(i + R) * m),
                             v2 = ldd(Vb + (long long)(i + 2 * R) * m), v3 = ldd(Vb + (long long)(i + 3 * R) * m);
                acc = fma(v0, ldd(rb + i), acc);
                acc = fma(v1, ldd(rb + i + R), acc);
                acc = fma(v2, ldd(rb + i + 2 * R), acc);
                acc = fma(v3, ldd(rb + i + 3 * R), acc);
            }
            for (; i < d; i += R) acc = fma(ldd(Vb + (long long)i * m), ldd(rb + i), acc);
        }
        part[t] = acc;
        __syncthreads();
        if (t < P) {
            double s = 0.0;
            for (int k = 0; k < R; ++k) s += part[k * P + t];
            r[b * m + c0 + t] = (T)s;
        }
        __syncthreads();
    }
}

// w[b * ldw + i] = sum_j V_b[i, j] s_b[j]; one CTA iteration per (sample, tile of 64 rows).  Panel by panel (<= 64
// columns), the tile's rows are staged into shared memory by loads that walk the panel's elements in memory order (for
// m <= 64 the tile is one contiguous block of V_b), then two threads per row sum the panel: the even thread the even
// columns, the odd thread the odd ones (pitch 66 doubles: the 16 lanes of a half-warp hit 16 different bank pairs).  Each
// thread adds its columns in ascending order over the panels; the row is the even half plus the odd half.
template <typename T>
__global__ void __launch_bounds__(kVbExpThreads)
vo_vb_expand_kernel(const T *__restrict__ V, const T *__restrict__ s, double *__restrict__ w, long long ldw, int d, int m,
                    long long B) {
    __shared__ __align__(16) double tile[kVbRows * kVbPitch];
    __shared__ double sp[kVbPanel];
    const int ntiles = (d + kVbRows - 1) / kVbRows;
    const int t = threadIdx.x, row = t >> 1, half = t & 1;
    for (long long job = blockIdx.x; job < B * ntiles; job += gridDim.x) {
        const long long b = job / ntiles;
        const int i0 = (int)(job - b * ntiles) * kVbRows, rows = min(kVbRows, d - i0);
        const T *Vt = V + (b * d + i0) * (long long)m;
        double acc = 0.0;
        for (int c0 = 0; c0 < m; c0 += kVbPanel) {
            const int P = min(kVbPanel, m - c0), n = rows * P;
            const int q = kVbExpThreads / P, rem = kVbExpThreads - q * P;   // (row, column) step of the element walk
            __syncthreads();   // the previous panel's reads of tile and sp are done
            if (t < P) sp[t] = ldd(s + b * m + c0 + t);
            int rr = t / P, cc = t - (t / P) * P;
#pragma unroll 8
            for (int e = t; e < n; e += kVbExpThreads) {
                tile[rr * kVbPitch + cc] = ldd(Vt + (long long)rr * m + c0 + cc);
                rr += q;
                cc += rem;
                if (cc >= P) { cc -= P; ++rr; }
            }
            __syncthreads();
            if (row < rows)
                for (int k = half; k < P; k += 2) acc = fma(tile[row * kVbPitch + k], sp[k], acc);
        }
        const double other = __shfl_xor_sync(0xffffffffu, acc, 1);
        if (row < rows && half == 0) w[b * ldw + i0 + row] = acc + other;
        // zero the row padding [d, ldw) as vo_expand_dmma_kernel does: no consumer may ever see stale workspace there
        if (i0 + rows == d && t < ldw - d) w[b * ldw + d + t] = 0.0;
    }
}

}  // namespace gpde

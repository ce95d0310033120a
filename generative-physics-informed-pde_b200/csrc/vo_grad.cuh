// Gradient of the virtual-observable residual r_b = V^T (K_fom(a_b) u~_b - f)_free with respect to the conductivity
// input a and the Dirichlet values g (sm_100a).  Included by vo.cu.
//
// With the incoming gradient gbar_r [B,m], w~_b = V gbar_r_b on the free dofs and 0 on the Dirichlet dofs (w = gbar_r V^T
// is produced by the expansion kernels of residual_T, launch_expand in vo.cu, and kept FP64 in the workspace).  K(a) is
// linear in a, so no solve is needed:
//   grad_a[b,p] = sum_{c : c2i(c) = p} w~_b[c]^T K_c u~_b[c]        ([c] = the cell's three dofs)
//   grad_g[b,k] = (K_cf(a_b) w~_b)_k                                 (the Dirichlet rows of K(a) applied to w~)
// The load vector does not enter either.  Every output is written by one thread with a fixed summation order: no atomics,
// and the results do not depend on the launch geometry.
#pragma once

namespace gpde {

// Plan data of the gradient kernels, built once in gpde_vo_plan_create.
struct VoGradDev {
    int n_inputs;
    const int *in_ptr;       // [n_inputs+1] cells of input p: entries in_ptr[p] .. in_ptr[p+1]-1 (ascending cell index)
    const int4 *cell_src;    // sources of the entry's three dofs (VoDev encoding: >= 0 free index, < 0 -(bc index)-1)
    const double *cell_K;    // [entries][9] the entry's unit-conductivity element matrix K_c, row-major
    VoCsrDev bc_rows;        // K_cf(a): rows = Dirichlet dofs (d = n_bc), columns = free dofs, (input, coef) terms
};

constexpr int kGradThreads = 256;

// u~ and w~ of one dof of sample b
template <typename T>
__device__ __forceinline__ void grad_dof(int src, const T *__restrict__ yb, const T *__restrict__ gb,
                                         const double *__restrict__ wb, double &u, double &wv) {
    if (src >= 0) {
        u = yb ? ldd(yb + src) : 0.0;
        wv = wb[src];
    } else {
        u = gb ? ldd(gb + (-src - 1)) : 0.0;
        wv = 0.0;
    }
}

// grad_a on the reference's pixel meshes (plans with grid.ok, vo.cu build_grid_plan): each pixel is two right triangles
// whose legs are the pixel's four edges (the hypotenuse does not couple), so with zero row sums
//   w~^T K_c u~ = -sum_{edges (i,j) of c} K_ij (w_i - w_j)(u_i - u_j)   and
//   grad_a[p] = kx (dw du on the bottom and top edges) + ky (dw du on the left and right edges),  kx = -chs, ky = -cvs.
// One thread per (sample, pixel column) marches over the node rows, holding the row below in registers; a warp reads 32
// consecutive nodes of a row (the right neighbour comes by shuffle), so y, w and a are read once per sample, row by row.
// Node (ix, r): ix = 0 / nx are the Dirichlet dofs 2r / 2r+1, the others free dof r (nx-1) + ix - 1.
template <typename T>
__global__ void __launch_bounds__(kGradThreads)
vo_grad_grid_kernel(int nx, int ny, long long in0, long long sy, double kx, double ky, const T *__restrict__ a,
                    long long a_stride, int a_is_log, const T *__restrict__ y, int d, const T *__restrict__ g,
                    long long g_stride, const double *__restrict__ w, long long ldw, T *__restrict__ grad_a, long long B) {
    const int lane = threadIdx.x & 31, ncol = nx - 1;
    const long long P = (long long)nx * ny, total = B * nx;
    const long long step = (long long)gridDim.x * kGradThreads;
    // warp-uniform loop: the shuffles below need every lane (a tail lane works on the last sample and stores nothing)
    for (long long base = (long long)blockIdx.x * kGradThreads + (threadIdx.x & ~31); base < total; base += step) {
        const long long idx = base + lane;
        const bool valid = idx < total;
        const long long b = valid ? idx / nx : B - 1;
        const int cx = (int)(idx - (long long)(idx / nx) * nx);
        const T *yb = y ? y + b * d : nullptr;
        const T *gb = g ? g + b * g_stride : nullptr;
        const double *wb = w + b * ldw;
        // (u, w) of nodes (cx, r) and (cx + 1, r)
        auto node_row = [&](int r, double &ul, double &wl, double &ur, double &wr) {
            if (cx == 0) {
                ul = gb ? ldd(gb + 2 * r) : 0.0;
                wl = 0.0;
            } else {
                const int i = r * ncol + cx - 1;
                ul = yb ? ldd(yb + i) : 0.0;
                wl = wb[i];
            }
            ur = __shfl_down_sync(0xffffffffu, ul, 1);
            wr = __shfl_down_sync(0xffffffffu, wl, 1);
            if (cx == nx - 1) {
                ur = gb ? ldd(gb + 2 * r + 1) : 0.0;
                wr = 0.0;
            } else if (lane == 31) {   // the neighbour belongs to the next warp: a cached re-read
                const int i = r * ncol + cx;
                ur = yb ? ldd(yb + i) : 0.0;
                wr = wb[i];
            }
        };
        double ul0, wl0, ur0, wr0;
        node_row(0, ul0, wl0, ur0, wr0);
#pragma unroll 2
        for (int r = 1; r <= ny; ++r) {
            double ul1, wl1, ur1, wr1;
            node_row(r, ul1, wl1, ur1, wr1);
            const double h = (wr0 - wl0) * (ur0 - ul0) + (wr1 - wl1) * (ur1 - ul1);
            const double v = (wl1 - wl0) * (ul1 - ul0) + (wr1 - wr0) * (ur1 - ur0);
            double ga = fma(kx, h, ky * v);
            const long long p = in0 + (long long)(r - 1) * sy + cx;
            if (a_is_log) ga *= exp(ldd(a + b * a_stride + p));
            if (valid) grad_a[b * P + p] = (T)ga;
            ul0 = ul1; wl0 = wl1; ur0 = ur1; wr0 = wr1;
        }
    }
}

// grad_a for every other plan: one thread per output (b, p) sums over the cells of input p.
template <typename T>
__global__ void __launch_bounds__(kGradThreads)
vo_grad_cells_kernel(VoGradDev G, const T *__restrict__ a, long long a_stride, int a_is_log, const T *__restrict__ y,
                     int d, const T *__restrict__ g, long long g_stride, const double *__restrict__ w, long long ldw,
                     T *__restrict__ grad_a, long long B) {
    const long long P = G.n_inputs, total = B * P;
    for (long long idx = (long long)blockIdx.x * kGradThreads + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * kGradThreads) {
        const long long b = idx / P;
        const int p = (int)(idx - b * P);
        const T *yb = y ? y + b * d : nullptr;
        const T *gb = g ? g + b * g_stride : nullptr;
        const double *wb = w + b * ldw;
        double acc = 0.0;
        const int e1 = G.in_ptr[p + 1];
        for (int e = G.in_ptr[p]; e < e1; ++e) {
            const int4 s = G.cell_src[e];
            const double *K = G.cell_K + 9ll * e;
            double u0, u1, u2, w0, w1, w2;
            grad_dof(s.x, yb, gb, wb, u0, w0);
            grad_dof(s.y, yb, gb, wb, u1, w1);
            grad_dof(s.z, yb, gb, wb, u2, w2);
            acc = fma(w0, fma(K[0], u0, fma(K[1], u1, K[2] * u2)), acc);
            acc = fma(w1, fma(K[3], u0, fma(K[4], u1, K[5] * u2)), acc);
            acc = fma(w2, fma(K[6], u0, fma(K[7], u1, K[8] * u2)), acc);
        }
        if (a_is_log) acc *= exp(ldd(a + b * a_stride + p));
        grad_a[idx] = (T)acc;
    }
}

// grad_g[b,k] = sum_j K_kj(a_b) w_b[j] over the Dirichlet row k of K(a), one thread per output.
template <typename T>
__global__ void __launch_bounds__(kGradThreads)
vo_grad_g_kernel(VoCsrDev C, const T *__restrict__ a, long long a_stride, int a_is_log, const double *__restrict__ w,
                 long long ldw, T *__restrict__ grad_g, long long B) {
    const long long nr = C.d, total = B * nr;
    for (long long idx = (long long)blockIdx.x * kGradThreads + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * kGradThreads) {
        const long long b = idx / nr;
        const int k = (int)(idx - b * nr);
        const T *ab = a + b * a_stride;
        const double *wb = w + b * ldw;
        double acc = 0.0;
        const int e1 = C.row_ptr[k + 1];
        for (int e = C.row_ptr[k]; e < e1; ++e) {
            double v = 0.0;
            const int t1 = C.term_ptr[e + 1];
            for (int t = C.term_ptr[e]; t < t1; ++t) {
                double av = ldd(ab + C.term_in[t]);
                if (a_is_log) av = exp(av);
                v = fma(av, C.term_coef[t], v);
            }
            acc = fma(v, wb[C.col[e]], acc);
        }
        grad_g[idx] = (T)acc;
    }
}

}  // namespace gpde

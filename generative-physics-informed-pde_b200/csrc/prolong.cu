// Prolongation y = W u and its transpose, W[d,n] = coarse P1 basis at the fine free nodes
// (bottleneck/components.py:298 einsum('sk,nk->ns', W, u); factories/model.py:140).
// The reference keeps W dense (d x n) and calls a GEMM; its rows have <= 3 non-zeros for P1, so it is
// held here as CSR (forward) + CSC (transpose) and applied as gathers -- the [B,d] output is written
// once, coalesced, and W itself stays in L1/L2.
#include "common.cuh"

#include <algorithm>

namespace gpde {
struct ProlongDev {
    int d, n;
    const int *row_ptr, *col;   // CSR
    const double *val;
    const int *col_ptr, *row;   // CSC
    const double *cval;
};
}  // namespace gpde

struct gpde_prolong_plan {
    gpde::ProlongDev dev;
    int device;
    std::vector<void *> allocs;
};

namespace gpde {

__device__ __forceinline__ double pld(const double *p) { return *p; }
__device__ __forceinline__ double pld(const float *p) { return (double)*p; }

template <typename T>
__global__ void prolong_apply_kernel(ProlongDev P, const T *__restrict__ u, T *__restrict__ y, long long B) {
    const long long total = B * (long long)P.d;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / P.d;
        const int i = (int)(idx - b * P.d);
        double acc = 0.0;
        const int t1 = P.row_ptr[i + 1];
        for (int t = P.row_ptr[i]; t < t1; ++t) acc = fma(P.val[t], pld(u + b * P.n + P.col[t]), acc);
        y[idx] = (T)acc;
    }
}

// one warp per (sample, coarse dof): reduce over the fine nodes in the hat function's support
template <typename T>
__global__ void prolong_apply_T_kernel(ProlongDev P, const T *__restrict__ gy, T *__restrict__ gu, long long B) {
    const int lane = threadIdx.x & 31;
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long total = B * (long long)P.n;
    for (long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < total; w += warps) {
        const long long b = w / P.n;
        const int k = (int)(w - b * P.n);
        double acc = 0.0;
        const int t1 = P.col_ptr[k + 1];
        for (int t = P.col_ptr[k] + lane; t < t1; t += 32) acc = fma(P.cval[t], pld(gy + b * P.d + P.row[t]), acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) gu[w] = (T)acc;
    }
}


// ---------------------------------------------------------------------------------------------------------------------
// Fused operator epilogue (SURVEY.md section 8 row f1): y = W u never reaches HBM.
//   L_b      = -1/2 sum_i [ 2 ls_i + ((Y_bi - (W u_b)_i) / sigma_i)^2 + log 2 pi ]      sigma_i = exp(ls_i)
//              = DiagonalGaussianLogLikelihood(Y_b, W u_b, 2 ls)  (bottleneck/utils.py:231-241) of the operator output
//              (bottleneck/components.py:296-298) as generative.py:438-439 evaluates it
//   gu_bk    = dL_b / du_bk      = sum_i W_ik (Y_bi - mu_bi) / sigma_i^2
//   gls_i    = d(sum_b L_b)/dls_i = sum_b (e_bi^2 - 1),   e = (Y - mu) / sigma
// Two launches over Y[B,d]: rows (thread per fine node, samples of the CTA's chunk in a loop: L and gls) and the weighted
// transposed prolongation (warp per (sample, coarse dof): gu).  L and gls are accumulated with FP64 atomics (a few per
// sample / per node and chunk).
constexpr int kLlThreads = 256, kLlSamples = 32;
constexpr double kLog2Pi = 1.8378770664093453;
// dynamic shared memory the loglik row kernel and the moments kernel may ask for (opted in above the 48 KB default)
constexpr size_t kMaxSmemBytes = 200 * 1024;

template <typename T>
__global__ void __launch_bounds__(kLlThreads)
prolong_loglik_rows_kernel(ProlongDev P, const T *__restrict__ u, const T *__restrict__ Y, const T *__restrict__ ls,
                           double *__restrict__ L, double *__restrict__ gls, long long B) {
    extern __shared__ double ll_smem[];
    double *us = ll_smem;                       // [kLlSamples][n]
    double *Ls = us + kLlSamples * P.n;         // [kLlSamples]
    const long long b0 = (long long)blockIdx.y * kLlSamples;
    const int nb = (int)min((long long)kLlSamples, B - b0);
    for (int idx = threadIdx.x; idx < nb * P.n; idx += kLlThreads) us[idx] = pld(u + b0 * P.n + idx);
    if (threadIdx.x < kLlSamples) Ls[threadIdx.x] = 0.0;
    __syncthreads();
    const int i = blockIdx.x * kLlThreads + threadIdx.x;
    const bool live = i < P.d;
    int t0 = 0, t1 = 0;
    double lsi = 0.0, inv = 0.0, gl = 0.0;
    if (live) {
        t0 = P.row_ptr[i]; t1 = P.row_ptr[i + 1];
        lsi = pld(ls + i);
        inv = exp(-lsi);
    }
    const int lane = threadIdx.x & 31;
    // 8 samples at a time: their Y values are fetched together (one global round trip per 8 samples, not one per sample:
    // small batches have too few CTAs to hide it), then reduced over the warp's rows
    for (int s0 = 0; s0 < nb; s0 += 8) {
        double yv[8];
#pragma unroll
        for (int w8 = 0; w8 < 8; ++w8) yv[w8] = (live && s0 + w8 < nb) ? pld(Y + (b0 + s0 + w8) * P.d + i) : 0.0;
#pragma unroll
        for (int w8 = 0; w8 < 8; ++w8) {
            const int sidx = s0 + w8;
            if (sidx >= nb) break;
            double term = 0.0;
            if (live) {
                double mu = 0.0;
                for (int t = t0; t < t1; ++t) mu = fma(P.val[t], us[sidx * P.n + P.col[t]], mu);
                const double e = (yv[w8] - mu) * inv;
                term = fma(e, e, 2.0 * lsi + kLog2Pi);
                gl += fma(e, e, -1.0);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) term += __shfl_xor_sync(0xffffffffu, term, o);
            if (lane == 0) atomicAdd(Ls + sidx, term);
        }
    }
    if (live && gls) atomicAdd(gls + i, gl);
    __syncthreads();
    if (threadIdx.x < nb) atomicAdd(L + b0 + threadIdx.x, -0.5 * Ls[threadIdx.x]);
}

// one warp per (sample, coarse dof): gu_bk = sum_{i in supp(k)} W_ik (Y_bi - (W u_b)_i) exp(-2 ls_i)
template <typename T>
__global__ void prolong_loglik_grad_kernel(ProlongDev P, const T *__restrict__ u, const T *__restrict__ Y,
                                           const T *__restrict__ ls, T *__restrict__ gu, long long B) {
    const int lane = threadIdx.x & 31;
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long total = B * (long long)P.n;
    for (long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < total; w += warps) {
        const long long b = w / P.n;
        const int k = (int)(w - b * P.n);
        const T *ub = u + b * P.n;
        double acc = 0.0;
        const int c1 = P.col_ptr[k + 1];
        for (int c = P.col_ptr[k] + lane; c < c1; c += 32) {
            const int i = P.row[c];
            double mu = 0.0;
            const int t1 = P.row_ptr[i + 1];
            for (int t = P.row_ptr[i]; t < t1; ++t) mu = fma(P.val[t], pld(ub + P.col[t]), mu);
            acc = fma(P.cval[c] * exp(-2.0 * pld(ls + i)), pld(Y + b * P.d + i) - mu, acc);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) gu[w] = (T)acc;
    }
}

// Monte-Carlo predictive moments of the operator output without the [N S, d] samples (generative.py:198-207 draws
// y_s = W u_s + sigma eps_s for S samples per data point and takes torch.mean / torch.std over them):
//   mean_i = W_i . ubar,   std_i = sqrt(W_i Cov_u W_i^T + sigma_i^2),   ubar / Cov_u = sample mean / unbiased covariance of u_s
// -- the same estimator with the noise eps integrated out (E over eps of the reference's unbiased sample variance).
// One CTA per data point: ubar and Cov_u (n x n) in shared memory, then one thread per fine node (<= 9 terms each).
template <typename T>
__global__ void __launch_bounds__(256)
prolong_moments_kernel(ProlongDev P, const T *__restrict__ u, const T *__restrict__ ls, T *__restrict__ y_mean,
                       T *__restrict__ y_std, int S) {
    extern __shared__ double mo_smem[];
    double *ubar = mo_smem;                 // [n]
    double *cov = ubar + P.n;               // [n][n]
    double *us = cov + P.n * P.n;           // [S][n] centred samples
    const long long nidx = blockIdx.x;
    const T *un = u + nidx * (long long)S * P.n;
    for (int k = threadIdx.x; k < P.n; k += blockDim.x) {
        double s = 0.0;
        for (int q = 0; q < S; ++q) s += pld(un + q * P.n + k);
        ubar[k] = s / S;
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < S * P.n; idx += blockDim.x) us[idx] = pld(un + idx) - ubar[idx % P.n];
    __syncthreads();
    const double denom = S > 1 ? 1.0 / (S - 1) : 0.0;
    for (int idx = threadIdx.x; idx < P.n * P.n; idx += blockDim.x) {
        const int a = idx / P.n, b = idx - a * P.n;
        double s = 0.0;
        for (int q = 0; q < S; ++q) s = fma(us[q * P.n + a], us[q * P.n + b], s);
        cov[idx] = s * denom;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < P.d; i += blockDim.x) {
        const int t0 = P.row_ptr[i], t1 = P.row_ptr[i + 1];
        double m = 0.0, v = 0.0;
        for (int t = t0; t < t1; ++t) {
            m = fma(P.val[t], ubar[P.col[t]], m);
            double r = 0.0;
            for (int t2 = t0; t2 < t1; ++t2) r = fma(P.val[t2], cov[P.col[t] * P.n + P.col[t2]], r);
            v = fma(P.val[t], r, v);
        }
        y_mean[nidx * P.d + i] = (T)m;
        y_std[nidx * P.d + i] = (T)sqrt(fmax(v, 0.0) + exp(2.0 * pld(ls + i)));
    }
}

template <typename T>
static int prolong_loglik(const gpde_prolong_plan *pl, const T *u, const T *Y, const T *ls, double *L, T *gu, double *gls,
                          int64_t B, gpde_stream_t stream) {
    if (!pl || B < 0) return fail(GPDE_ERR_ARG, "prolong_loglik: bad argument");
    if (B > 0 && (!u || !Y || !ls || !L)) return fail(GPDE_ERR_ARG, "prolong_loglik: null argument");
    const size_t smem = sizeof(double) * ((size_t)kLlSamples * pl->dev.n + kLlSamples);
    if (B > 0 && smem > kMaxSmemBytes)
        return fail(GPDE_ERR_SIZE, "prolong_loglik: %d samples x %d dofs do not fit in shared memory", kLlSamples,
                    pl->dev.n);
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    // gls sums over the batch: an empty batch (a rank without samples) contributes zeros, not whatever gls held
    if (gls) GPDE_CUDA_OK(cudaMemsetAsync(gls, 0, sizeof(double) * (size_t)pl->dev.d, st));
    if (B == 0) return GPDE_OK;
    auto rows = prolong_loglik_rows_kernel<T>;
    if (smem > 48 * 1024) GPDE_CUDA_OK(cudaFuncSetAttribute(rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    GPDE_CUDA_OK(cudaMemsetAsync(L, 0, sizeof(double) * (size_t)B, st));
    const dim3 grid((unsigned)((pl->dev.d + kLlThreads - 1) / kLlThreads), (unsigned)((B + kLlSamples - 1) / kLlSamples));
    rows<<<grid, kLlThreads, smem, st>>>(pl->dev, u, Y, ls, L, gls, B);
    if (gu) {
        const long long total = B * (long long)pl->dev.n;   // warps
        const unsigned g2 = (unsigned)std::min<long long>((total + 7) / 8, (long long)sm_count(pl->device) * 16);
        prolong_loglik_grad_kernel<T><<<g2, 256, 0, st>>>(pl->dev, u, Y, ls, gu, B);
    }
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

template <typename T>
static int prolong_moments(const gpde_prolong_plan *pl, const T *u, const T *ls, T *y_mean, T *y_std, int64_t N, int S,
                           gpde_stream_t stream) {
    if (!pl || N < 0 || S < 1) return fail(GPDE_ERR_ARG, "prolong_moments: bad argument");
    if (N == 0) return GPDE_OK;
    if (!u || !ls || !y_mean || !y_std) return fail(GPDE_ERR_ARG, "prolong_moments: null argument");
    const size_t smem = sizeof(double) * ((size_t)pl->dev.n * (1 + pl->dev.n) + (size_t)S * pl->dev.n);
    if (smem > kMaxSmemBytes) return fail(GPDE_ERR_SIZE, "prolong_moments: %d samples x %d dofs do not fit in shared memory", S, pl->dev.n);
    DeviceGuard guard(pl->device);
    auto kern = prolong_moments_kernel<T>;
    GPDE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)N, 256, smem, (cudaStream_t)stream>>>(pl->dev, u, ls, y_mean, y_std, S);
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

template <typename T>
static cudaError_t track_p(gpde_prolong_plan *pl, const T **dst, const std::vector<T> &src) {
    T *p = nullptr;
    cudaError_t e = upload(&p, src);
    if (p) pl->allocs.push_back((void *)p);
    *dst = p;
    return e;
}

template <typename T>
static int prolong_apply(const gpde_prolong_plan *pl, const T *u, T *y, int64_t B, gpde_stream_t stream, bool transpose) {
    if (!pl || B < 0) return fail(GPDE_ERR_ARG, "prolong_apply: bad argument");
    if (B == 0) return GPDE_OK;
    if (!u || !y) return fail(GPDE_ERR_ARG, "prolong_apply: null argument");
    DeviceGuard guard(pl->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int nsm = sm_count(pl->device);
    if (!transpose) {
        const long long total = B * (long long)pl->dev.d;
        const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, (long long)nsm * 16);
        prolong_apply_kernel<T><<<grid, 256, 0, st>>>(pl->dev, u, y, B);
    } else {
        const long long total = B * (long long)pl->dev.n;   // warps
        const unsigned grid = (unsigned)std::min<long long>((total + 7) / 8, (long long)nsm * 16);
        prolong_apply_T_kernel<T><<<grid, 256, 0, st>>>(pl->dev, u, y, B);
    }
    GPDE_CUDA_OK(cudaGetLastError());
    return GPDE_OK;
}

}  // namespace gpde

using namespace gpde;

extern "C" {

int gpde_prolong_plan_create(gpde_prolong_plan **plan, int d, int n, const double *W, int device) {
    if (!plan || !W || d <= 0 || n <= 0) return fail(GPDE_ERR_ARG, "prolong_plan_create: bad argument");
    std::vector<int> row_ptr(d + 1, 0), col, col_ptr(n + 1, 0), row;
    std::vector<double> val, cval;
    for (int i = 0; i < d; ++i) {
        for (int k = 0; k < n; ++k) {
            const double v = W[(size_t)i * n + k];
            if (v != 0.0) {
                col.push_back(k);
                val.push_back(v);
            }
        }
        row_ptr[i + 1] = (int)col.size();
    }
    for (int k = 0; k < n; ++k) {
        for (int i = 0; i < d; ++i) {
            const double v = W[(size_t)i * n + k];
            if (v != 0.0) {
                row.push_back(i);
                cval.push_back(v);
            }
        }
        col_ptr[k + 1] = (int)row.size();
    }
    gpde_prolong_plan *pl = new gpde_prolong_plan();
    pl->device = device;
    DeviceGuard guard(device);
    ProlongDev &D = pl->dev;
    D.d = d; D.n = n;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = track_p(pl, &D.row_ptr, row_ptr);
    if (e == cudaSuccess) e = track_p(pl, &D.col, col);
    if (e == cudaSuccess) e = track_p(pl, &D.val, val);
    if (e == cudaSuccess) e = track_p(pl, &D.col_ptr, col_ptr);
    if (e == cudaSuccess) e = track_p(pl, &D.row, row);
    if (e == cudaSuccess) e = track_p(pl, &D.cval, cval);
    if (e != cudaSuccess) {
        gpde_prolong_plan_destroy(pl);
        return fail(GPDE_ERR_CUDA, "prolong_plan_create: upload failed: %s", cudaGetErrorString(e));
    }
    *plan = pl;
    return GPDE_OK;
}

int gpde_prolong_plan_destroy(gpde_prolong_plan *pl) {
    if (!pl) return GPDE_OK;
    DeviceGuard guard(pl->device);
    for (void *p : pl->allocs) cudaFree(p);
    delete pl;
    return GPDE_OK;
}

int gpde_prolong_apply_f64(const gpde_prolong_plan *pl, const double *u, double *y, int64_t B, gpde_stream_t s) {
    return prolong_apply<double>(pl, u, y, B, s, false);
}
int gpde_prolong_apply_T_f64(const gpde_prolong_plan *pl, const double *gy, double *gu, int64_t B, gpde_stream_t s) {
    return prolong_apply<double>(pl, gy, gu, B, s, true);
}
int gpde_prolong_loglik_f64(const gpde_prolong_plan *pl, const double *u, const double *Y, const double *ls, double *L,
                            double *gu, double *gls, int64_t B, gpde_stream_t s) {
    return prolong_loglik<double>(pl, u, Y, ls, L, gu, gls, B, s);
}
int gpde_prolong_loglik_f32(const gpde_prolong_plan *pl, const float *u, const float *Y, const float *ls, double *L,
                            float *gu, double *gls, int64_t B, gpde_stream_t s) {
    return prolong_loglik<float>(pl, u, Y, ls, L, gu, gls, B, s);
}
int gpde_prolong_moments_f64(const gpde_prolong_plan *pl, const double *u, const double *ls, double *y_mean, double *y_std,
                             int64_t N, int S, gpde_stream_t s) {
    return prolong_moments<double>(pl, u, ls, y_mean, y_std, N, S, s);
}
int gpde_prolong_moments_f32(const gpde_prolong_plan *pl, const float *u, const float *ls, float *y_mean, float *y_std,
                             int64_t N, int S, gpde_stream_t s) {
    return prolong_moments<float>(pl, u, ls, y_mean, y_std, N, S, s);
}
int gpde_prolong_apply_f32(const gpde_prolong_plan *pl, const float *u, float *y, int64_t B, gpde_stream_t s) {
    return prolong_apply<float>(pl, u, y, B, s, false);
}
int gpde_prolong_apply_T_f32(const gpde_prolong_plan *pl, const float *gy, float *gu, int64_t B, gpde_stream_t s) {
    return prolong_apply<float>(pl, gy, gu, B, s, true);
}

}  // extern "C"

// Structured-grid virtual-observable residual kernel (sm_100a).  Included by vo.cu.
//
// When the fine mesh is the reference's own (pixels of two P1 triangles on an nx x ny grid,
// factories/model.py:130-133; Dirichlet data on the left/right edges, LinearEllipticFactories.py:173-179,
// 239-281) and the conductivity comes per pixel (bottleneck/utils.py:41-98), K_fom(a) is a 5-point
// operator: the coupling of two horizontally adjacent nodes is chs * (a[pixel below] + a[pixel above]),
// of two vertically adjacent ones cvs * (a[pixel left] + a[pixel right]); the hypotenuse couplings of
// right-angled P1 triangles vanish.  gpde_vo_plan_create verifies this against the element data it is
// given and otherwise leaves the generic kernels (vo_fused.cuh / version 1) in charge.
//
//   r[b,:] = V^T (K_fom(a_b) u~_b - f)_free        (VirtualObservables.py:61-69, 662, 990)
//
// A CTA of 16 warps marches over the node rows bottom to top; warp (group, strip) = 8 samples x 16 node columns, lane
// (s = lane/4, k = lane%4) owns 4 columns of sample s and keeps the row below in registers; flux form
// S_i = rh (Fh_right - Fh_left) + (Fv_up - Fv_down), rho_i = cvs * S_i - f_i; the 4 values a lane produces ARE its A
// fragments of four mma.sync.m8n8k4.f64 k-steps (M = 8 samples, K = 4 lanes' columns, N = 8 columns of V), the B
// fragments come from a fragment-packed V row in shared memory.  The inner loop carries no generality:
//   * nx in {16, 32, 64, 128} pixels per row and an even number of pixel rows (build_grid_plan in vo.cu), no load vector
//     (LinearEllipticFactories.py:165-171 is the zero load; a plan with one is served here only when the call ignores it);
//   * exactly one lane per warp row touches the left Dirichlet column and one the right one: two selects per
//     row instead of per-column category decoding; no column masks; first and last node row peeled;
//   * a stage = 2 node rows; every thread copies the same 4 + 4 16-byte pieces per stage (one piece position in
//     4 samples), addresses advance by a constant: ~35 instructions per thread and stage;
//   * B fragments two at a time (LDS.128 from a pair-packed V row);
//   * m = 8 NT + NX: the NX (0 or 1) columns past the last full n-tile go through DFMA with one accumulator per
//     lane (m = 25: 3 DMMA tiles + 1 DFMA column instead of 4 tiles: -12 % FP64-pipe cycles per node row).
//   * one a / y ring per sample group (own mbarriers), the packed V rows in a ring of their own; exp() by a 256-entry
//     2^(j/256) table + degree-4 polynomial with constant-bank coefficients; a_is_log, the rho output and a strided y
//     are template parameters (the kernel's time follows its instruction count and is sensitive to the register
//     allocation: every variant gets its own).
// Shared memory: 2 a/y stages | 2-3 V stages | barriers | exp table; the a/y stages are zero-initialised once so that the
// few halo reads that fall outside a sample's rows see finite numbers.
//   * the I/O element types are template parameters (TA: conductivities and Dirichlet values, TY: y, TR: result): FP32 I/O
//     stages the rows as floats (half the copies, half the shared memory) and converts when a lane reads its values; the
//     arithmetic is FP64 in every variant (the reference's model dtype is float32, factories/model.py:181,224).
//   * the packed V rows travel through a ring of 2-3 stages filled by bulk copies; the refill is event-driven (the warp whose
//     arrival completes a slot's empty phase issues the next copy), the strips are rotated over the schedulers by the group
//     index, a CTA may take fewer samples than it has slots (the launcher balances the last wave over the SMs);
//   * SPLIT: small batches as thread-block clusters that cut the node rows; WT (KS > 0): the transposed application
//     q = K_ff(a) (V s) with the rows of V s produced by DMMAs inside the kernel (see the comments at the kernel).
#pragma once
#include "exp256.cuh"

namespace gpde {

struct Grid2Dev {
    int nx, ny, ncol, lognx;
    int nstrips, lognstrips, groups;
    long long in0, sy;       // conductivity entry of pixel (cx, cy) = in0 + cy * sy + cx
    double rh, scale;
    int a_pitch, y_pitch;    // elements (of TA / TY) per sample inside a stage
    int y_off, v_off;        // byte offsets inside a stage
    int stage_bytes, v_row_bytes;   // one a/y stage (all samples of the CTA); one packed V row
    int nvs;                        // V stages in the ring (2 or 3)
    int spc;                        // samples a CTA takes (<= 8 groups): group i gets [i spc / groups, (i + 1) spc / groups)
    int wait_first;                 // programmatic dependent of a kernel this one does not know: griddepcontrol.wait first
};

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16_u32(unsigned smem_dst, const void *gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}

__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    const unsigned addr = smem_u32(bar);
    unsigned done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)   // (a suspend-time hint made wake-ups ~10x slower on B200: measured, not used)
            : "memory");
        if (!done) __nanosleep(40);
    } while (!done);
}
// global -> shared bulk copy (TMA engine, 1-D); bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void cp_async8_u32(unsigned smem_dst, const void *gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async4_u32(unsigned smem_dst, const void *gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ bool mbar_test(unsigned long long *bar, unsigned parity) {
    unsigned done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return done != 0;
}
// DMMA under a warp-uniform predicate (straight-line code: a skipped link of an accumulator chain costs an issue slot, no
// pipe time and no latency; as branches around the DMMAs the same skipping made the WT variant 16 % slower)
__device__ __forceinline__ void dmma884_if(unsigned on, double &d0, double &d1, double a, double b) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.u32 p, %4, 0;\n\t"
        "@p mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n\t}"
        : "+d"(d0), "+d"(d1)
        : "d"(a), "d"(b), "r"(on));
}
__device__ __forceinline__ double2 lds128(unsigned addr) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ double lds64(unsigned addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}

__device__ __forceinline__ float lds32f(unsigned addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ float4 lds128f(unsigned addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
// one staged element as a double
template <typename T> __device__ __forceinline__ double lds_elem(unsigned addr);
template <> __device__ __forceinline__ double lds_elem<double>(unsigned addr) { return lds64(addr); }
template <> __device__ __forceinline__ double lds_elem<float>(unsigned addr) { return (double)lds32f(addr); }

// |x| <= 700 (false for NaN / inf) from the high word alone: integer pipe, no FP64 compare
__device__ __forceinline__ int exp_arg_hi(double x) { return __double2hiint(x) & 0x7fffffff; }
constexpr int kExpHiMax = 0x4085e000;   // high word of 700.0

// V[d,m] row-major -> per node row t: [strip q][n-tile tt < NT][half ph < 2][lane][2], then [strip q][k][4] (NX = 1 only),
// then one 32-bit mask per strip (8 words, 32 bytes).
//   tile tt, half ph, element h: k-step jj = 2 ph + h; lane = 4 n + kk holds V[t*ncol + 16 q + 4 kk + jj][8 tt + n];
//   extra column: V[t*ncol + 16 q + 4 k + j][8 NT]     (0 outside the matrix)
//   mask of (t, q): bit tt set <=> the 16 x 8 block of V behind n-tile tt has a non-zero entry, bit 7 <=> the extra column
//   has one.  The residual kernel skips the B-fragment loads and the four DMMAs of a tile whose block is all zero
//   (exact: it only drops products with 0): V = W of the coarse-grained-residual sampler (VirtualObservables.py:297-321)
//   has <= 4 non-zero columns per block (P1 hat functions of the coarse mesh), i.e. 1-2 of its 3-4 tiles.
constexpr int kGrid2MaskBytes = 32;
template <typename TV>
__global__ void vo_grid2_pack_kernel(Grid2Dev G, const TV *__restrict__ V, int m, int NT, int NX,
                                     double *__restrict__ Vp) {
    // programmatic dependent launch: the residual kernel may start its prologue (shared-memory setup, first a / y
    // stages) now; it waits for this grid (griddepcontrol.wait) before it touches the packed rows
    asm volatile("griddepcontrol.launch_dependents;");
    // one warp per (node row t, strip q): it writes the strip's NT tiles (128 doubles each, 4 per lane), the extra column
    // and -- from the values it has just seen -- the strip's mask word.  All loads of a warp are issued before its first
    // store (NT <= 4 tiles unrolled): the launch sits on the critical path of a residual call, and a loop over the tiles
    // with its stores in between waits out one load round trip per tile.
    const int per_strip = 4 * NT * 32, per_row = G.v_row_bytes / 8, main = G.nstrips * per_strip;
    const int data = main + (NX ? G.nstrips * 16 : 0);     // doubles of a row before the masks
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long w = warp; w < (long long)(G.ny + 1) * 8; w += nwarps) {
        const int t = (int)(w >> 3), q = (int)(w & 7);
        double *row = Vp + (long long)t * per_row;
        unsigned bits = 0;
        if (q < G.nstrips) {
            const TV *Vt = V + (long long)t * G.ncol * m;
            double v[4][4], vx = 0.0;
#pragma unroll
            for (int tt = 0; tt < 4; ++tt)
#pragma unroll
                for (int it = 0; it < 4; ++it) {
                    const int e = it * 32 + lane;                       // [half ph][lane ln][h]
                    const int h = e & 1, ln = (e >> 1) & 31, ph = e >> 6;
                    const int c = 16 * q + 4 * (ln & 3) + 2 * ph + h, col = 8 * tt + (ln >> 2);
                    v[tt][it] = (tt < NT && c < G.ncol && col < m) ? (double)Vt[(long long)c * m + col] : 0.0;
                }
            if (NX) {
                const int c = 16 * q + lane, col = 8 * NT;               // [k][j] = column 16 q + 4 k + j: lanes 0..15
                vx = (lane < 16 && c < G.ncol && col < m) ? (double)Vt[(long long)c * m + col] : 0.0;
            }
#pragma unroll
            for (int tt = 0; tt < 4; ++tt)
                if (tt < NT) {
                    bool nz = false;
#pragma unroll
                    for (int it = 0; it < 4; ++it) {
                        row[q * per_strip + tt * 128 + it * 32 + lane] = v[tt][it];
                        nz |= v[tt][it] != 0.0;
                    }
                    if (__any_sync(0xffffffffu, nz)) bits |= 1u << tt;
                }
            if (NX) {
                if (lane < 16) row[main + q * 16 + lane] = vx;
                if (__any_sync(0xffffffffu, vx != 0.0)) bits |= 0x80u;
            }
        }
        if (lane == 0) reinterpret_cast<unsigned *>(row + data)[q] = bits;
    }
}

// Transposed application (WT variant of the kernel below): V[d,mw] row-major -> per node row t the B fragments of
// w_row = s V_row^T (mma.sync.m8n8k4.f64: 8 samples x 8 nodes, contraction over the weighting functions):
//   [strip q][n-tile nt < 2][k-step ks < KS][lane]:  V[t*ncol + 16 q + 8 nt + lane / 4][4 ks + lane % 4]  (0 outside V)
// then one 32-bit mask per strip (8 words): bit nt * KS + ks set <=> that 8-node x 4-function block of V has a non-zero
// entry.  The kernel skips the fragment load and the DMMA of an empty block (exact: it only drops products with 0): the
// coarse-grained-residual sampler's V = W (VirtualObservables.py:297-321) has 4 non-zero functions per node, i.e. 2 - 4 of
// the 7 k-steps of m = 25.
template <typename TV>
__global__ void vo_grid2_pack_t_kernel(Grid2Dev G, const TV *__restrict__ V, int mw, int KS, double *__restrict__ Vp) {
    const int per_row = G.v_row_bytes / 8, data = per_row - kGrid2MaskBytes / 8;
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long w = warp; w < (long long)(G.ny + 1) * 8; w += nwarps) {     // one warp per (node row t, strip slot q)
        const int t = (int)(w >> 3), q = (int)(w & 7);
        double *row = Vp + (long long)t * per_row;
        unsigned bits = 0;
        if (q < G.nstrips) {
            for (int c2 = 0; c2 < 2 * KS; ++c2) {                               // c2 = nt * KS + ks
                const int nt = c2 / KS, ks = c2 - nt * KS;
                const int c = 16 * q + 8 * nt + (lane >> 2), j = 4 * ks + (lane & 3);
                const double v = (c < G.ncol && j < mw) ? (double)V[((long long)t * G.ncol + c) * mw + j] : 0.0;
                row[(q * 2 * KS + c2) * 32 + lane] = v;
                if (__any_sync(0xffffffffu, v != 0.0)) bits |= 1u << c2;
            }
        }
        if (lane == 0) reinterpret_cast<unsigned *>(row + data)[q] = bits;
    }
}

// the B fragments and DMMAs of the n-tiles named by the compile-time MASK (straight-line code per mask value: the tiles'
// accumulator chains are independent and interleave)
template <int NT, int MASK, typename LoadPair>
__device__ __forceinline__ void grid2_contract_tiles(double (&acc)[NT][2], const double (&Sv)[4], LoadPair load_pair) {
    double bf[NT][4];
#pragma unroll
    for (int tt = 0; tt < NT; ++tt)
        if (MASK >> tt & 1) {
            const double2 v0 = load_pair(2 * tt), v1 = load_pair(2 * tt + 1);
            bf[tt][0] = v0.x; bf[tt][1] = v0.y; bf[tt][2] = v1.x; bf[tt][3] = v1.y;
        }
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
#pragma unroll
        for (int tt = 0; tt < NT; ++tt)
            if (MASK >> tt & 1) dmma884(acc[tt][0], acc[tt][1], Sv[jj], bf[tt][jj]);
}
template <int NT, typename LoadPair>
__device__ __forceinline__ void grid2_contract(unsigned msk, double (&acc)[NT][2], const double (&Sv)[4], LoadPair load_pair) {
    switch (msk & ((1u << NT) - 1u)) {
#define GPDE_G2_CASE(M) case M: if constexpr (M < (1 << NT)) grid2_contract_tiles<NT, M>(acc, Sv, load_pair); break;
        GPDE_G2_CASE(1) GPDE_G2_CASE(2) GPDE_G2_CASE(3) GPDE_G2_CASE(4) GPDE_G2_CASE(5) GPDE_G2_CASE(6) GPDE_G2_CASE(7)
        GPDE_G2_CASE(8) GPDE_G2_CASE(9) GPDE_G2_CASE(10) GPDE_G2_CASE(11) GPDE_G2_CASE(12) GPDE_G2_CASE(13)
        GPDE_G2_CASE(14) GPDE_G2_CASE(15)
#undef GPDE_G2_CASE
        default: break;
    }
}

// SPLIT (small batches, launched as thread-block clusters): the C CTAs of a cluster share one block of samples and cut the
// node rows into C contiguous ranges of stages.  A range that does not start at the bottom first replays the stage before
// it with the contraction switched off (that rebuilds the marching state: previous node row, previous pixel row, vertical
// fluxes); each CTA reduces its strips as usual, the partial results meet in rank order through distributed shared memory
// on rank 0.  The cut depends only on the number of sample blocks of the call, never on a sample's position in the batch.
// WT (KS > 0; rho variant only): the transposed application q = K_ff(a) (V s) = Gamma^T s (VirtualObservables.py:663) in ONE
// kernel -- "accumulating the residual gradient directly": the node rows of w = s V^T are not staged from global memory
// but PRODUCED by the group's warps, a stage ahead of their use, straight into the y slots of the stage: a warp forms its
// 8 samples x 16 columns of a node row with 2 x KS DMMAs (A fragments = the samples' s, KS k-steps, in registers for the
// whole kernel; B fragments from the packed V^T rows of the V ring) and its D fragments go to shared memory as 16-byte
// pieces (row pitch nx inside a slot); the group's full barrier counts the warps' arrivals beside the threads' cp.async
// arrivals of the conductivity rows.  w [B,d] (134 MB written and read back at config 2) never exists.  In this variant
// `g` / `g_stride` carry s [B,mw] and mw (the Dirichlet data of the transposed application are zero), `y` is unused.
template <int NT, int NX, bool RHO, bool YS, bool ALOG, typename TA = double, typename TY = double, typename TR = double,
          bool SPLIT = false, int KS = 0>
__global__ void __launch_bounds__(512, 1)
vo_grid2_kernel(Grid2Dev G, const TA *__restrict__ a, long long a_stride, int a_is_log,
                const TY *__restrict__ y, long long y_stride_arg, const TA *__restrict__ g, long long g_stride,
                const double *__restrict__ Vp, int m, TR *__restrict__ r, long long B) {
    // y_stride = elements between the rows of consecutive samples in y: d for a contiguous [B,d]; only the YS variant
    // takes it from its argument (the expansion kernel of residual_T pads the rows of w to a multiple of 4 doubles):
    // one more live value shifts the register allocation of the other variants by ~3 % (measured A/B on one box)
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int kThreads = 512, kWarps = 16;
    constexpr bool WT = KS > 0;
    static_assert(!WT || (RHO && !YS && !SPLIT && sizeof(TY) == 8), "WT: rho variant with FP64 y slots");
    constexpr int NP = 2 * NT;                      // B-fragment pairs per strip and node row
    constexpr int EA = (int)sizeof(TA), EY = (int)sizeof(TY);   // bytes per staged element
    // shared memory: 2 a/y stages | nvs V stages | barriers | exp table
    const int v_bytes = 2 * G.v_row_bytes;          // one V stage = 2 packed rows
    unsigned char *v_base = smem_raw + 2 * (size_t)G.stage_bytes;
    unsigned long long *full_ay = reinterpret_cast<unsigned long long *>(v_base + (size_t)G.nvs * v_bytes);   // [group][2]
    unsigned long long *empty_ay = full_ay + 2 * kWarps;
    unsigned long long *full_v = empty_ay + 2 * kWarps;                                                         // [nvs <= 4]
    unsigned long long *empty_v = full_v + 4;
    double *tab = reinterpret_cast<double *>(empty_v + 4);
    const unsigned sm0 = smem_u32(smem_raw);
    const unsigned tab32 = smem_u32(tab);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // group and strip of this warp.  The warps of a sample group sit on ONE scheduler (warp % 4 for four groups): every
    // scheduler then hosts all strips -- their work differs from node row to node row with the non-zero tiles of V -- and a
    // warp that waits for its group leaves its issue slots to the warps it waits for.  (Groups of consecutive warps, one
    // strip per scheduler: 58.1 us at config 2; the same rotated by the group index: 57.0 us; this: 56.6 us and the
    // log-input variant 79.6 instead of 82.4 us -- A/Bs on one box each.)
    const int grp = warp & (G.groups - 1), q = warp >> (4 - G.lognstrips);
    const int s = lane >> 2, k = lane & 3;
    const int S = 8 * G.groups;
    const int sl = grp * 8 + s;
    // Samples of the CTA: its 8-sample groups are filled with gsz <= 8 samples each (rows s >= gsz of the group's DMMA tile
    // idle), spc = sum of the sizes.  The launcher picks spc so that the CTAs of the last wave spread over all SMs (4096
    // samples: 147 CTAs of 28 instead of 128 of 32 on 148 SMs); a sample's arithmetic does not depend on its slot.
    const int lgg = 4 - G.lognstrips;               // log2(groups)
    const int goff = (grp * G.spc) >> lgg, gsz = (((grp + 1) * G.spc) >> lgg) - goff;
    unsigned crank = 0, csize = 1;                  // rank in the cluster and its size (SPLIT only)
    if constexpr (SPLIT) {
        asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
        asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(csize));
    }
    const long long cta_b0 = (long long)(SPLIT ? blockIdx.x / csize : blockIdx.x) * G.spc;
    const long long grp_b0 = cta_b0 + goff;         // first sample of this warp's group
    const bool b_valid = s < gsz && grp_b0 + s < B;
    const long long b = b_valid ? grp_b0 + s : B - 1;
    const int ncol = G.ncol, nx = G.nx, ny = G.ny;
    const long long d = (long long)ncol * (ny + 1);
    const long long y_stride = YS ? y_stride_arg : d;
    const int c0 = 16 * q + 4 * k;
    const int n_stages = ny >> 1;
    // stages [ts_base, ts_base + n_local) of this CTA; with SPLIT the first one of ranks > 0 is the replayed stage
    const int s_lo = SPLIT ? (int)((long long)n_stages * crank / csize) : 0;
    const int s_hi = SPLIT ? (int)((long long)n_stages * (crank + 1) / csize) : n_stages;
    const bool warm = SPLIT && crank > 0;
    const int ts_base = warm ? s_lo - 1 : s_lo;
    const int n_local = s_hi - ts_base;
    const int gthreads = 32 * G.nstrips;            // threads of one sample group (= 2 nx)
    const bool is_left = c0 == 0, is_right = c0 == nx - 4;
    const TY *yb = y + b * y_stride;
    const TA *gp = (!WT && g && (is_left || is_right)) ? g + b * g_stride + (is_right ? 1 : 0) : nullptr;
    // Launched as a programmatic dependent of whatever the stream ran before (prepacked weights): nothing from global
    // memory is read before that grid has completed; only the launch overlaps it.  (After the packing kernel of the same
    // call, its prerequisites completed before it started, and only the packed rows wait for it: see below.)
    if (G.wait_first) asm volatile("griddepcontrol.wait;" ::: "memory");
    // node row 0 of this lane comes straight from global memory: requested here, consumed after the set-up below (one
    // exposed DRAM round trip less per CTA: in the profile of a one-wave launch 3.5 % of the warp samples sat behind it)
    double r0[4] = {0.0, 0.0, 0.0, 0.0}, r0l = 0.0, r0r = 0.0, r0g = 0.0;
    if (!WT && !warm) {
        if (gp) r0g = (double)__ldg(gp);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (c0 + j < ncol) r0[j] = (double)__ldg(yb + c0 + j);
        if (!is_left) r0l = (double)__ldg(yb + c0 - 1);
        if (c0 + 4 < ncol) r0r = (double)__ldg(yb + c0 + 4);
    }

    // ---- zero the stages (halo reads past a sample's rows must see finite numbers), barriers, exp table
    {
        const int n16 = (2 * G.stage_bytes) >> 4;   // a / y stages only: every byte of a V stage is overwritten
        for (int i = tid; i < n16; i += kThreads)
            asm volatile("st.shared.v2.f64 [%0], {%1,%1};" ::"r"(sm0 + 16 * i), "d"(0.0) : "memory");
    }
    if (tid == 0) {
        for (int i = 0; i < 2 * G.groups; ++i) {
            mbar_init(full_ay + i, gthreads + (WT ? G.nstrips : 0));
            mbar_init(empty_ay + i, G.nstrips);
        }
        for (int i = 0; i < G.nvs; ++i) {
            mbar_init(full_v + i, 1);
            mbar_init(empty_v + i, kWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if constexpr (ALOG) {
        if (tid < 256) tab[tid] = kExp256Tab[tid];
    }
    __syncthreads();

    // ---- staging.  Every sample group (8 samples, nstrips warps) runs its OWN two-stage ring of a / y rows with its
    // own barriers, so the groups drift apart and the four warps of a scheduler (one per group) sit in different
    // phases of the row (exp / fluxes / DMMA / waiting); only the packed V rows are shared by the CTA (ring of nvs
    // stages, copied by thread 0).  A sample's two rows of a stage are 2 nx E / 16 pieces of 16 bytes (E = element
    // size): the 2 nx threads of a group copy piece (tg mod pieces) of samples (tg / pieces) + (16 / E) i, i < E / 2
    // (FP64: 4 pieces per thread and array, samples 2 apart; FP32: 2 pieces, samples 4 apart).
    const int tg = q * 32 + lane;                   // thread index inside the sample group
    constexpr int NIA = EA / 2, SSA = 16 / EA, NIY = EY / 2, SSY = 16 / EY;
    const int lpa = G.lognx - (EA == 8 ? 0 : 1), lpy = G.lognx - (EY == 8 ? 0 : 1);   // log2(pieces per sample)
    const int j0a = tg >> lpa, j0 = tg >> lpy;      // first sample (inside the group) this thread copies of a / of y
    const int piece_a = tg & ((1 << lpa) - 1), smp0a = 8 * grp + j0a;
    const int piece = tg & ((1 << lpy) - 1), smp0 = 8 * grp + j0;                      // y
    int nva = 0, nv = 0;
#pragma unroll
    for (int i = 0; i < NIA; ++i) nva += (j0a + SSA * i < gsz && grp_b0 + j0a + SSA * i < B) ? 1 : 0;
#pragma unroll
    for (int i = 0; i < NIY; ++i) nv += (j0 + SSY * i < gsz && grp_b0 + j0 + SSY * i < B) ? 1 : 0;
    // pixel rows 2 ts, 2 ts + 1 of a sample are one block of 2 nx elements (lowest address first)
    const long long a_adv = 2 * EA * G.sy, a_smp = SSA * a_stride * EA;
    const char *a_src = reinterpret_cast<const char *>(a + (grp_b0 + j0a) * a_stride + G.in0 + (G.sy > 0 ? 0 : G.sy)) + 16 * piece_a +
                        (SPLIT ? ts_base * a_adv : 0);
    const unsigned a_dst = smp0a * G.a_pitch * EA + 16 * piece_a, a_dsmp = SSA * G.a_pitch * EA;
    // node rows 2 ts + 1, 2 ts + 2: 2 ncol elements starting on an element boundary; copied from the enclosing
    // 16-byte boundary.  The phase y_sig (in elements) is the same for the samples of a thread (they are 16 / E apart).
    // FP64: it is the same for all stages too (a stage advances by 16 ncol bytes); FP32: a stage advances by 8 ncol
    // bytes with ncol odd, so the phase alternates between y_sig and y_sig ^ 2 from stage to stage
    const char *y_row1 = reinterpret_cast<const char *>(y + (grp_b0 + j0) * y_stride + ncol + (SPLIT ? 2 * ts_base * ncol : 0));
    int y_sig = (int)(((unsigned long long)y_row1 / EY) & (16 / EY - 1));
    const char *y_src = y_row1 - EY * y_sig + 16 * piece;
    const long long y_adv = 2 * EY * ncol, y_smp = SSY * y_stride * EY;
    // FP64: slot of sample sl starts at (sl * y_pitch + 2 * ((sl >> 1) & 1) + 2) doubles; (smp0 + 2 i) >> 1 has the parity of i.
    // FP32: at (sl * y_pitch + 4) floats; the phases of consecutive samples differ (d is odd) and y_pitch = 4 mod 8, so the
    // 8 samples x 4 lanes of a warp read 32 different banks
    const unsigned y_dst = G.y_off + (smp0 * G.y_pitch + (EY == 8 ? 2 : 4)) * EY + 16 * piece, y_dsmp = SSY * G.y_pitch * EY;
    // FP64: the last piece is needed only with phase 1; FP32: the window of 2 nx floats always ends in the last piece, and
    // with phase 3 one more float follows it
    const bool y_last_piece = piece == (1 << lpy) - 1;
    const bool y_piece_ok = EY == 8 ? (!y_last_piece || y_sig) : true;
    // the last piece of the batch's last sample would read past the tensor: copied element-wise instead
    // (FP32: only when the stage's phase leaves part of the piece outside, decided per stage)
    const bool y_tail = (EY == 8 ? y_sig != 0 : true) && y_last_piece && nv > 0 && grp_b0 + j0 + SSY * (nv - 1) == B - 1;
    unsigned long long *my_full = full_ay + 2 * grp, *my_empty = empty_ay + 2 * grp;

    auto issue_stage = [&](int ts, int slot) {
        const unsigned sb = sm0 + slot * G.stage_bytes;
#pragma unroll
        for (int i = 0; i < NIA; ++i)
            if (i < nva) cp_async16_u32(sb + a_dst + i * a_dsmp, a_src + i * a_smp);
        if (!WT && y_piece_ok) {
            const int nvy = nv - ((y_tail && ts == n_stages - 1 && (EY == 8 || y_sig < 2)) ? 1 : 0);
            if constexpr (EY == 8) {
#pragma unroll
                for (int i = 0; i < NIY; ++i)
                    if (i < nvy) cp_async16_u32(sb + y_dst + i * y_dsmp + 16 * (i & 1), y_src + i * y_smp);
                if (nvy != nv) cp_async8_u32(sb + y_dst + (nv - 1) * y_dsmp + 16 * ((nv - 1) & 1), y_src + (nv - 1) * y_smp);
            } else {
#pragma unroll
                for (int i = 0; i < NIY; ++i)
                    if (i < nvy) cp_async16_u32(sb + y_dst + i * y_dsmp, y_src + i * y_smp);
                if (nvy != nv)      // the y_sig + 2 floats of the piece that belong to the tensor
                    for (int e = 0; e < y_sig + 2; ++e)
                        cp_async4_u32(sb + y_dst + (nv - 1) * y_dsmp + 4 * e, y_src + (nv - 1) * y_smp + 4 * e);
                if (y_last_piece && y_sig == 3) {   // the float behind the window (last node of the stage's second row)
#pragma unroll
                    for (int i = 0; i < NIY; ++i)
                        if (i < nv) cp_async4_u32(sb + y_dst + i * y_dsmp + 16, y_src + i * y_smp + 16);
                }
            }
        }
        asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(my_full + slot)) : "memory");
        a_src += a_adv;
        y_src += y_adv;
        if constexpr (EY == 4) {   // next stage: phase y_sig ^ 2, source re-aligned to its 16-byte boundary
            y_src -= 4 * ((y_sig ^ 2) - y_sig);
            y_sig ^= 2;
        }
    };
    issue_stage(ts_base, 0);
    if (n_local > 1) issue_stage(ts_base + 1, 1);

    // Packed V rows -> ring of nvs V stages (forward: packed rows 2 ts, 2 ts + 1, the rows whose residual the stage completes;
    // WT: rows 2 ts + 1, 2 ts + 2, the node rows the stage brings in).  Thread 0 primes the ring; afterwards the refill is
    // EVENT-DRIVEN: the warp whose arrival completes a slot's empty phase copies stage j + nvs into it at once -- whoever
    // observes the completed phase first, elected in stage order through the shared counter v_next.  (Until late in round 2
    // thread 0 refilled at the top of its own iterations: it found the slot "just about to be released" and so ran one stage
    // ahead instead of nvs - 1; the warps slept 13 times per stage waiting for V rows.  61.8 -> 59.4 us at config 2.)
    const unsigned v_next32 = tab32 + 256 * 8;          // shared-memory address of the counter
    auto copy_v = [&](int j, int slot_) {
        mbar_arrive_expect_tx(full_v + slot_, (unsigned)v_bytes);
        bulk_g2s(v_base + (size_t)slot_ * v_bytes,
                 reinterpret_cast<const char *>(Vp) + (size_t)(2 * (ts_base + j) + (WT ? 1 : 0)) * G.v_row_bytes, (unsigned)v_bytes,
                 full_v + slot_);
    };
    if ((!RHO || WT) && tid == 0) {
        asm volatile("griddepcontrol.wait;" ::: "memory");   // the packing kernel's rows (no-op without a dependent launch)
        int j = 0;
        for (; j < G.nvs && j < n_local; ++j) copy_v(j, j);
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(v_next32), "r"(j) : "memory");
    }
    // release of V stage j_done (slot v_slot_, parity v_par_) by this warp's lane 0
    auto release_v = [&](int j_done, int v_slot_, unsigned v_par_) {
        mbar_arrive(empty_v + v_slot_);
        const int j = j_done + G.nvs;
        if (j < n_local && mbar_test(empty_v + v_slot_, v_par_)) {
            int cur;
            do {   // (cur < j: the copy of the stage before is still being issued)
                asm volatile("atom.shared.cas.b32 %0, [%1], %2, %3;" : "=r"(cur) : "r"(v_next32), "r"(j), "r"(j + 1) : "memory");
            } while (cur < j);
            if (cur == j) copy_v(j, v_slot_);
        }
    };

    // ---- per-lane constants of the consumer
    const int sig_b = WT ? 0 : (int)(((unsigned long long)(y + (grp_b0 + s) * y_stride + ncol) / EY) & (16 / EY - 1));
    // byte offsets inside a stage of this lane's first column: y row 2 ts + 1, pixel row 2 ts, V pairs
    // (WT: the rows are produced in place, always at an even offset, and read back as 16-byte pieces: consecutive samples
    //  2 doubles apart modulo 4 make the quarter-warps of those loads conflict-free)
    const unsigned y_lane = G.y_off + (sl * G.y_pitch + (EY == 8 ? 2 * (WT ? (sl & 1) : ((sl >> 1) & 1)) + 2 : 4) + sig_b + c0) * EY;
    const int y_lane_odd = EY == 4 ? 4 * ((sig_b ^ 2) - sig_b) : 0;   // FP32: odd (global) stages sit at phase sig_b ^ 2
    const unsigned a_lane0 = (sl * G.a_pitch + c0) * EA + (G.sy > 0 ? 0 : nx * EA);   // pixel row 2 ts
    const unsigned a_lane1 = (sl * G.a_pitch + c0) * EA + (G.sy > 0 ? nx * EA : 0);   // pixel row 2 ts + 1
    const unsigned v_lane = (q * NP * 32 + lane) * 16;                       // inside a V stage
    const unsigned x_lane = G.nstrips * NP * 512 + (q * 4 + k) * 32;
    const int mask_dbl = (G.v_row_bytes - kGrid2MaskBytes) >> 3;          // doubles of a packed row before its masks
    const unsigned m_lane = G.v_row_bytes - kGrid2MaskBytes + 4 * q;
    const unsigned row_bytes = WT ? nx * 8 : ncol * EY;      // WT: the produced rows sit at pitch nx inside a slot
    const double rh = G.rh;
    const bool rho_wide = RHO && !(m & 1) && !(reinterpret_cast<unsigned long long>(r) & 15ull);

    double acc[NT][2], accx = 0.0;
#pragma unroll
    for (int tt = 0; tt < NT; ++tt) acc[tt][0] = acc[tt][1] = 0.0;
    double uc[4], ulc, urc, ap[5], fvp[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) fvp[j] = 0.0;
#pragma unroll
    for (int j = 0; j < 5; ++j) ap[j] = 0.0;
    // WT: this lane's A fragments (sample s of the group, weighting functions 4 ks + k) and the producer of a stage's rows
    double af[WT ? KS : 1];
    const unsigned wt_dst = y_lane - 16 * k;                       // columns 16 q + 2 k, + 1 of row 0 of the slot
    const unsigned vt_lane = (unsigned)(q * 2 * (WT ? KS : 1)) * 256 + lane * 8;   // inside a packed V^T row
    int v_slot = 0;                  // V stage being consumed and the parity of its full barrier
    unsigned v_par = 0;
    // rows of one stage: 2 node rows x 2 n-tiles = 4 independent accumulator chains of KS DMMAs, interleaved; the values
    // stay in registers (cw) until the stage's slot is free, so the contraction overlaps the wait for the group's other
    // warps; the V stage is released as soon as its fragments have been read
    auto wt_compute = [&](double (&cw)[8], int j_stage) {
        if constexpr (WT) {
            mbar_wait(full_v + v_slot, v_par);
            const unsigned vb = smem_u32(v_base) + v_slot * v_bytes + vt_lane;
            unsigned mk[2];                  // non-zero blocks of this strip in the stage's two rows (bit nt * KS + ks)
#pragma unroll
            for (int rr = 0; rr < 2; ++rr)
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(mk[rr]) : "r"(smem_u32(v_base) + v_slot * v_bytes + rr * G.v_row_bytes + m_lane));
#pragma unroll
            for (int i = 0; i < 8; ++i) cw[i] = 0.0;
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
                for (int rr = 0; rr < 2; ++rr) {
                    dmma884_if(mk[rr] & (1u << ks), cw[4 * rr], cw[4 * rr + 1], af[ks], lds64(vb + rr * G.v_row_bytes + ks * 256));
                    dmma884_if(mk[rr] & (1u << (KS + ks)), cw[4 * rr + 2], cw[4 * rr + 3], af[ks],
                               lds64(vb + rr * G.v_row_bytes + (KS + ks) * 256));
                }
            }
            __syncwarp();
            if (lane == 0) release_v(j_stage, v_slot, v_par);
            if (++v_slot == G.nvs) { v_slot = 0; v_par ^= 1; }
        }
    };
    auto wt_store = [&](unsigned sb_dst, int slot_i, const double (&cw)[8]) {
        if constexpr (WT) {
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
                const unsigned dst = sb_dst + wt_dst + rr * row_bytes;
                asm volatile("st.shared.v2.f64 [%0], {%1,%2};" ::"r"(dst), "d"(cw[4 * rr]), "d"(cw[4 * rr + 1]) : "memory");
                asm volatile("st.shared.v2.f64 [%0], {%1,%2};" ::"r"(dst + 64), "d"(cw[4 * rr + 2]), "d"(cw[4 * rr + 3]) : "memory");
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(my_full + slot_i);
        }
    };
    if constexpr (WT) {
#pragma unroll
        for (int ks = 0; ks < KS; ++ks)
            af[ks] = (b_valid && 4 * ks + k < (int)g_stride) ? (double)__ldg(g + b * g_stride + 4 * ks + k) : 0.0;
        // node row 0: B fragments from packed row 0 in global memory, through the y slot of stage 0 (its left / right
        // neighbours belong to other warps of the group), before the stage's own rows are produced
        {
            const double *vg = Vp + (vt_lane >> 3);
            double c00 = 0.0, c01 = 0.0, c10 = 0.0, c11 = 0.0;
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {      // (zero blocks contribute zeros: no need for the masks here)
                dmma884(c00, c01, af[ks], __ldg(vg + ks * 32));
                dmma884(c10, c11, af[ks], __ldg(vg + (KS + ks) * 32));
            }
            asm volatile("st.shared.v2.f64 [%0], {%1,%2};" ::"r"(sm0 + wt_dst), "d"(c00), "d"(c01) : "memory");
            asm volatile("st.shared.v2.f64 [%0], {%1,%2};" ::"r"(sm0 + wt_dst + 64), "d"(c10), "d"(c11) : "memory");
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) uc[j] = lds64(sm0 + y_lane + 8 * j);
        ulc = is_left ? 0.0 : lds64(sm0 + y_lane - 8);
        urc = lds64(sm0 + y_lane + 32);
        if (is_right) uc[3] = 0.0;
        __syncthreads();
        {
            double cw[8];
            wt_compute(cw, 0);
            wt_store(sm0, 0, cw);
            if (n_local > 1) {
                wt_compute(cw, 1);
                wt_store(sm0 + G.stage_bytes, 1, cw);
            }
        }
    } else
    // node row 0 straight from global memory (a range that starts higher up gets its state from the replayed stage)
    if (SPLIT && warm) {
#pragma unroll
        for (int j = 0; j < 4; ++j) uc[j] = 0.0;
        ulc = urc = 0.0;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) uc[j] = r0[j];
        ulc = is_left ? r0g : r0l;
        urc = r0r;
        if (is_right) uc[3] = r0g;
    }
    // Dirichlet values of the first stage's node rows 2 ts + 1, 2 ts + 2
    double gn0 = gp ? (double)__ldg(gp + 2 * (2 * ts_base + 1)) : 0.0, gn1 = gp ? (double)__ldg(gp + 2 * (2 * ts_base + 2)) : 0.0;

    // one node row: new row (un, an) in, residual of the row below (uc between ap and an) out
    auto node_row = [&](const double (&un)[4], double unl, double unr, const double (&an)[5], unsigned v_addr,
                        unsigned x_addr, unsigned msk_s, const double *v_glob, int t_out) {
        double fh[5];
        fh[0] = (ap[0] + an[0]) * (uc[0] - ulc);
#pragma unroll
        for (int j = 1; j < 4; ++j) fh[j] = (ap[j] + an[j]) * (uc[j] - uc[j - 1]);
        fh[4] = (ap[4] + an[4]) * (urc - uc[3]);
        double Sv[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double fv = (an[j] + an[j + 1]) * (un[j] - uc[j]);
            Sv[j] = fma(rh, fh[j + 1] - fh[j], fv - fvp[j]);
            fvp[j] = fv;
        }
        if (is_right) Sv[3] = 0.0;
        if constexpr (RHO) {
            if (b_valid) {
                TR *dst = r + b * (long long)m + (long long)t_out * ncol + c0;
                if (sizeof(TR) == 8 && rho_wide) {
                    // even row pitch, 16-byte aligned rows: ncol is odd, so this lane's 4 values start on a 16-byte boundary
                    // in even node rows and 8 bytes past one in odd rows -- 2 or 3 stores instead of 4
                    double *dd = reinterpret_cast<double *>(dst);
                    const double s0 = G.scale * Sv[0], s1 = G.scale * Sv[1], s2 = G.scale * Sv[2], s3 = G.scale * Sv[3];
                    if (!(t_out & 1)) {
                        *reinterpret_cast<double2 *>(dd) = make_double2(s0, s1);
                        if (!is_right) *reinterpret_cast<double2 *>(dd + 2) = make_double2(s2, s3);
                        else dd[2] = s2;
                    } else {
                        dd[0] = s0;
                        *reinterpret_cast<double2 *>(dd + 1) = make_double2(s1, s2);
                        if (!is_right) dd[3] = s3;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 3; ++j) dst[j] = (TR)(G.scale * Sv[j]);
                    if (!is_right) dst[3] = (TR)(G.scale * Sv[3]);
                }
            }
        } else {
            if (v_glob) {   // last node row: packed V row from global memory
                const unsigned msk = __ldg(reinterpret_cast<const unsigned *>(v_glob + mask_dbl) + q);
                const double2 *vg = reinterpret_cast<const double2 *>(v_glob) + q * NP * 32 + lane;
                grid2_contract<NT>(msk, acc, Sv, [&](int p) { return __ldg(vg + p * 32); });
                if constexpr (NX > 0) {
                    if (msk & 0x80u) {
                        const double2 *xp = reinterpret_cast<const double2 *>(v_glob) + G.nstrips * NP * 32 + (q * 4 + k) * 2;
                        const double2 x0 = __ldg(xp), x1 = __ldg(xp + 1);
                        accx = fma(Sv[0], x0.x, accx);
                        accx = fma(Sv[1], x0.y, accx);
                        accx = fma(Sv[2], x1.x, accx);
                        accx = fma(Sv[3], x1.y, accx);
                    }
                }
            } else {
                grid2_contract<NT>(msk_s, acc, Sv, [&](int p) { return lds128(v_addr + p * 512); });
                if constexpr (NX > 0) {
                    if (msk_s & 0x80u) {
                        const double2 x0 = lds128(x_addr), x1 = lds128(x_addr + 16);
                        accx = fma(Sv[0], x0.x, accx);
                        accx = fma(Sv[1], x0.y, accx);
                        accx = fma(Sv[2], x1.x, accx);
                        accx = fma(Sv[3], x1.y, accx);
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) uc[j] = un[j];
        ulc = unl; urc = unr;
#pragma unroll
        for (int j = 0; j < 5; ++j) ap[j] = an[j];
    };

    for (int lt = 0; lt < n_local; ++lt) {
        const int ts = ts_base + lt;
        const int slot = lt & 1;
        const unsigned par = (lt >> 1) & 1;
        const unsigned sb = sm0 + slot * G.stage_bytes;
        const unsigned vb = smem_u32(v_base) + v_slot * v_bytes;
        mbar_wait(my_full + slot, par);
        if (!RHO) mbar_wait(full_v + v_slot, v_par);
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const unsigned ya = sb + y_lane + rr * row_bytes + (EY == 4 && (SPLIT ? (ts & 1) : slot) ? y_lane_odd : 0);
            unsigned msk_rr = 0;
            if constexpr (!RHO) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(msk_rr) : "r"(vb + m_lane + rr * G.v_row_bytes));
            double un[4], unl, unr, an[5];
            unl = lds_elem<TY>(ya - EY);
            if constexpr (WT) {
                const double2 u01 = lds128(ya), u23 = lds128(ya + 16);
                un[0] = u01.x; un[1] = u01.y; un[2] = u23.x; un[3] = u23.y;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) un[j] = lds_elem<TY>(ya + EY * j);
            }
            unr = lds_elem<TY>(ya + 4 * EY);
            const double gv = rr ? gn1 : gn0;
            if (is_left) unl = gv;
            if (is_right) un[3] = gv;
            if (SPLIT && warm && lt == 0) {
                // replayed stage: its first node row only becomes the "row below"; its second one runs with the contraction
                // off (empty mask), which leaves the marching state as if the rows below had been processed
                if (rr == 0) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) uc[j] = un[j];
                    ulc = unl; urc = unr;
                    continue;
                }
                msk_rr = 0;
            }
            const unsigned aa = sb + (rr ? a_lane1 : a_lane0);
            if constexpr (EA == 8) {
                const double2 p0 = lds128(aa), p1 = lds128(aa + 16);
                an[0] = p0.x; an[1] = p0.y; an[2] = p1.x; an[3] = p1.y;
                an[4] = lds64(aa + 32);
            } else {
                const float4 p0 = lds128f(aa);
                an[0] = (double)p0.x; an[1] = (double)p0.y; an[2] = (double)p0.z; an[3] = (double)p0.w;
                an[4] = (double)lds32f(aa + 16);
            }
            if constexpr (ALOG) {
                int hmax = exp_arg_hi(an[4]);
#pragma unroll
                for (int j = 0; j < 4; ++j) hmax = max(hmax, exp_arg_hi(an[j]));
#pragma unroll
                for (int j = 0; j < 5; ++j) an[j] = exp_tab256c(an[j], tab32);
                if (hmax > kExpHiMax) {   // |x| > 700, inf or NaN somewhere in the warp's row (rare): libm exp() on the
                                          // values re-read from shared memory, so the common path keeps no copies
#pragma unroll
                    for (int j = 0; j < 5; ++j) an[j] = exp(lds_elem<TA>(aa + EA * j));
                }
            }
            if (rr == 1) {
                // the stage's a / y rows are in registers now: release the slot BEFORE the second row's arithmetic, so that
                // the group's other warps find it free when they come to refill it (with the release at the end of the stage
                // 10 % of the warp samples sat in that wait: 67.4 -> 62.6 us A/B on one box; refilling here as well, half a
                // stage earlier, is slower again: 64.8 us)
                __syncwarp();
                if (lane == 0) mbar_arrive(my_empty + slot);
            }
            node_row(un, unl, unr, an, vb + v_lane + rr * G.v_row_bytes, vb + x_lane + rr * G.v_row_bytes, msk_rr, nullptr,
                     2 * ts + rr);
        }
        if (gp && ts + 1 < n_stages) {       // Dirichlet values of the next stage's rows 2 ts + 3, 2 ts + 4
            gn0 = (double)__ldg(gp + 2 * (2 * ts + 3));
            gn1 = (double)__ldg(gp + 2 * (2 * ts + 4));
        }
        __syncwarp();
        if (lane == 0) {
            if (!RHO) release_v(lt, v_slot, v_par);
        }
        if constexpr (!WT) {
            if (++v_slot == G.nvs) { v_slot = 0; v_par ^= 1; }
        }
        if (lt + 2 < n_local) {
            double cw[WT ? 8 : 1];
            if constexpr (WT) wt_compute(cw, lt + 2);
            mbar_wait(my_empty + slot, par);
            issue_stage(ts + 2, slot);
            if constexpr (WT) wt_store(sb, slot, cw);
        }
    }
    // ---- last node row (ny): no pixel row above (SPLIT: the top range only)
    if (!SPLIT || crank == csize - 1) {
        if (!RHO) asm volatile("griddepcontrol.wait;" ::: "memory");   // packed row ny is read with plain loads
        const double un[4] = {0.0, 0.0, 0.0, 0.0}, an[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
        node_row(un, 0.0, 0.0, an, 0u, 0u, 0u,
                 RHO ? nullptr : reinterpret_cast<const double *>(reinterpret_cast<const char *>(Vp) + (size_t)ny * G.v_row_bytes),
                 ny);
    }

    if constexpr (RHO) {
        const int pad = m - (int)d;   // zero the K padding [d, m) of this CTA's rows
        for (int idx = tid; idx < G.spc * pad; idx += kThreads) {   // (samples cta_b0 .. cta_b0 + spc - 1, whatever their slots)
            const int si = idx / pad, c = idx - si * pad;
            if (cta_b0 + si < B) r[(cta_b0 + si) * (long long)m + d + c] = (TR)0;
        }
        return;
    }
    // ---- sum the strips' partial tiles and store r = cvs * sum   (stage memory is free now)
    constexpr int NW = NT * 8 + 2 * NX;   // doubles per (sample, strip) record
    if constexpr (NX > 0) {
        accx += __shfl_xor_sync(0xffffffffu, accx, 1);
        accx += __shfl_xor_sync(0xffffffffu, accx, 2);
    }
    __syncthreads();
    double *red = reinterpret_cast<double *>(smem_raw);   // [groups][nstrips][8 samples][NW]
    {
        double *dst = red + (((size_t)grp * G.nstrips + q) * 8 + s) * NW;
#pragma unroll
        for (int tt = 0; tt < NT; ++tt) {
            dst[tt * 8 + 2 * k] = acc[tt][0];
            dst[tt * 8 + 2 * k + 1] = acc[tt][1];
        }
        if (NX > 0 && k == 0) dst[NT * 8] = accx;
    }
    __syncthreads();
    constexpr int MC = NT * 8 + NX;
    if constexpr (SPLIT) {
        // this range's partial result of the CTA's samples, behind ``red``; rank 0 adds the ranks' partials in rank order
        double *part = red + (size_t)kWarps * 8 * NW;      // [S][MC]
        for (int idx = tid; idx < S * MC; idx += kThreads) {
            const int si = idx / MC, col = idx - si * MC;
            const int gi = si >> 3, ss = si & 7;
            double v = 0.0;
            for (int qq = 0; qq < G.nstrips; ++qq) v += red[(((size_t)gi * G.nstrips + qq) * 8 + ss) * NW + col];
            part[idx] = v;
        }
        asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
        if (crank == 0) {
            const unsigned part32 = smem_u32(part);
            for (int idx = tid; idx < S * MC; idx += kThreads) {
                const int si = idx / MC, col = idx - si * MC;
                const int gi = si >> 3, ss = si & 7;
                const int go = (gi * G.spc) >> lgg, gs = (((gi + 1) * G.spc) >> lgg) - go;
                const long long bs = cta_b0 + go + ss;
                if (col < m && ss < gs && bs < B) {
                    double v = 0.0;
                    for (unsigned c = 0; c < csize; ++c) {
                        unsigned remote;
                        double pv;
                        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(part32 + 8u * idx), "r"(c));
                        asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(pv) : "r"(remote) : "memory");
                        v += pv;
                    }
                    r[bs * m + col] = (TR)(G.scale * v);
                }
            }
        }
        // nobody leaves (and frees its shared memory) before rank 0 has read it
        asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    } else {
        for (int idx = tid; idx < S * MC; idx += kThreads) {
            const int si = idx / MC, col = idx - si * MC;
            const int gi = si >> 3, ss = si & 7;
            const int go = (gi * G.spc) >> lgg, gs = (((gi + 1) * G.spc) >> lgg) - go;
            const long long bs = cta_b0 + go + ss;
            if (col < m && ss < gs && bs < B) {
                double v = 0.0;
                for (int qq = 0; qq < G.nstrips; ++qq) v += red[(((size_t)gi * G.nstrips + qq) * 8 + ss) * NW + col];
                r[bs * m + col] = (TR)(G.scale * v);
            }
        }
    }
}

}  // namespace gpde

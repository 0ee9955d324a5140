// Saved PCA model: per-variant loadings of a fitted context and scoring of new cohorts against them (include/vpca.h,
// DESIGN.md 3.7).
//
// Expanding the cross count X_pf = sum_v x_pv x_fv of the projection formula (eig.cu, proj_*) over variants gives the
// same coordinate from per-variant quantities of the fitted panel:
//   L_vc = sum_f x_fv u_fc (loadings),  n_v = sum_f x_fv (carriers),  a_c = sum_f u_fc,  b_c = sum_f (rs_f / N) u_fc
//   T_pc = sum_v x_pv L_vc,  r_p = sum_v x_pv n_v (= rs_p, exact),  y_pc = (((T_pc - (r_p / N) a_c) - b_c) + mean a_c) / l_c
// Both passes read the encoded chunks the existing encoders produce (panel layout, ceil(nv / P) panels of `rows` x P
// cells) and need no tensor cores: every cell costs k FP64 FMAs, so the loadings pass (N x V cells) and the scoring pass
// (M x V cells) are bound by the FP64 rate or by the HBM read of the cells, whichever is larger (tools/model_bench.py).
// Every reduction has a fixed order (no atomics), so repeated calls are bit-identical.
#include <cuda_runtime.h>

#include <algorithm>

#include "vpca_internal.h"

namespace vpca {
namespace {

// Cell values as integers (multiplicities): int8 as is, bf16 bits through float, e2m1 code 2 m -> m.
template <int BITS>
__device__ __forceinline__ int cell_value(uint32_t raw) {
    if constexpr (BITS == 8) return (int)(int8_t)(raw & 0xFFu);
    else if constexpr (BITS == 16) return (int)__uint_as_float((raw & 0xFFFFu) << 16);
    else return (int)((raw & 0xFu) >> 1);
}

// 4 consecutive cells starting at cell index `cell` (a multiple of 4).
template <int BITS>
__device__ __forceinline__ void load4(const uint8_t* __restrict__ x, int64_t cell, int (&v)[4]) {
    if constexpr (BITS == 8) {
        const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(x + cell));
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = cell_value<8>(w >> (8 * j));
    } else if constexpr (BITS == 16) {
        const uint2 w = __ldg(reinterpret_cast<const uint2*>(x + cell * 2));
        v[0] = cell_value<16>(w.x); v[1] = cell_value<16>(w.x >> 16);
        v[2] = cell_value<16>(w.y); v[3] = cell_value<16>(w.y >> 16);
    } else {
        const uint32_t w = __ldg(reinterpret_cast<const uint16_t*>(x + cell / 2));
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = cell_value<4>(w >> (4 * j));
    }
}

// 16 consecutive cells starting at cell index `cell` (a multiple of 16).
template <int BITS>
__device__ __forceinline__ void load16(const uint8_t* __restrict__ x, int64_t cell, int (&v)[16]) {
    if constexpr (BITS == 8) {
        const uint4 w = __ldg(reinterpret_cast<const uint4*>(x + cell));
        const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = cell_value<8>(ws[j >> 2] >> (8 * (j & 3)));
    } else if constexpr (BITS == 16) {
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(x + cell * 2));
        const uint4 b = __ldg(reinterpret_cast<const uint4*>(x + cell * 2) + 1);
        const uint32_t ws[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = cell_value<16>(ws[j >> 1] >> (16 * (j & 1)));
    } else {
        const uint2 w = __ldg(reinterpret_cast<const uint2*>(x + cell / 2));
        const uint32_t ws[2] = {w.x, w.y};
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = cell_value<4>(ws[j >> 3] >> (4 * (j & 7)));
    }
}

// ---- loadings ----------------------------------------------------------------------------------------------------
// One thread = 4 consecutive variants x KC columns [c0, c0 + KC) of u.  The loop runs over the fitted rows f = 0..N-1
// in ascending order and adds x_fv u_fc with one FMA each (x in {0, 1, 2, ...}: the product is exact), so the value of a
// variant's loadings depends on f alone -- not on the chunk, the route or the thread that computes it.  A row whose 4
// cells are all zero adds nothing and is skipped (rare variants make most cells zero).  u is read with warp-uniform
// addresses (one broadcast per column and row).
constexpr int kLoadThreads = 128;

template <int BITS, int KC>
__global__ void __launch_bounds__(kLoadThreads) model_loadings_kernel(const uint8_t* __restrict__ x, int64_t nv,
                                                                      int64_t panel, int rows, int n_fit,
                                                                      const double* __restrict__ U, int k, int c0,
                                                                      double* __restrict__ L, int32_t* __restrict__ carriers) {
    const int64_t v0 = ((int64_t)blockIdx.x * kLoadThreads + threadIdx.x) * 4;
    if (v0 >= nv) return;
    const int64_t pnl = v0 / panel;
    const uint8_t* __restrict__ xp = x;
    const int64_t base = pnl * (int64_t)rows * panel + (v0 - pnl * panel);   // cell (row 0, v0)
    const int kc = min(KC, k - c0);
    double acc[4][KC];
    int cnt[4] = {0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int c = 0; c < KC; ++c) acc[j][c] = 0.0;
    constexpr int kAhead = 4;   // rows loaded before the first of them is used
    for (int f0 = 0; f0 < n_fit; f0 += kAhead) {
        int xv[kAhead][4];
#pragma unroll
        for (int i = 0; i < kAhead; ++i) {
            if (f0 + i < n_fit) load4<BITS>(xp, base + (int64_t)(f0 + i) * panel, xv[i]);
            else xv[i][0] = xv[i][1] = xv[i][2] = xv[i][3] = 0;
        }
#pragma unroll
        for (int i = 0; i < kAhead; ++i) {
            if ((xv[i][0] | xv[i][1] | xv[i][2] | xv[i][3]) == 0) continue;
            const int f = f0 + i;
            double u[KC];
#pragma unroll
            for (int c = 0; c < KC; ++c) u[c] = c < kc ? __ldg(U + (size_t)(c0 + c) * n_fit + f) : 0.0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                cnt[j] += xv[i][j];
                const double xd = (double)xv[i][j];
#pragma unroll
                for (int c = 0; c < KC; ++c) acc[j][c] = __fma_rn(xd, u[c], acc[j][c]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int64_t v = v0 + j;
        if (v >= nv) break;
#pragma unroll
        for (int c = 0; c < KC; ++c)
            if (c < kc) L[v * k + c0 + c] = acc[j][c];
        if (c0 == 0) carriers[v] = cnt[j];
    }
}

template <int KC>
cudaError_t loadings_launch(const void* d_x, int elem_bits, int64_t nv, int64_t panel, int rows, int n_fit,
                            const double* d_u, int k, double* d_L, int32_t* d_carriers, cudaStream_t stream) {
    const int64_t blocks = ((nv + 3) / 4 + kLoadThreads - 1) / kLoadThreads;
    const uint8_t* x = static_cast<const uint8_t*>(d_x);
    for (int c0 = 0; c0 < k; c0 += KC) {
        if (elem_bits == 8)
            model_loadings_kernel<8, KC><<<(unsigned)blocks, kLoadThreads, 0, stream>>>(x, nv, panel, rows, n_fit, d_u, k, c0,
                                                                                       d_L, d_carriers);
        else if (elem_bits == 16)
            model_loadings_kernel<16, KC><<<(unsigned)blocks, kLoadThreads, 0, stream>>>(x, nv, panel, rows, n_fit, d_u, k, c0,
                                                                                        d_L, d_carriers);
        else
            model_loadings_kernel<4, KC><<<(unsigned)blocks, kLoadThreads, 0, stream>>>(x, nv, panel, rows, n_fit, d_u, k, c0,
                                                                                       d_L, d_carriers);
    }
    return cudaGetLastError();
}

// ---- scoring -----------------------------------------------------------------------------------------------------
// One thread = one study sample p, KC columns.  The variants of a chunk are cut into stages of kStage variants inside
// one panel; a block stages the model rows of a stage in shared memory (gathered through m(v); rows with m(v) = -1 are
// zero), then every thread walks its sample's cells of the stage in ascending v, 16 cells per load (one 16-byte load of
// its sample row for int8).  The stages of a chunk are dealt to `ranges` blocks in contiguous runs; each block writes
// one partial per sample, and model_fold_kernel adds the partials of the ranges in ascending order to the accumulator.
// Stages, ranges and both orders depend only on (nv, panel, m): the same chunk always gives the same bits.
constexpr int kScoreThreads = 128;
constexpr int kStage = 512;
constexpr int kMaxRangeBlocks = 2048;   // ranges x sample groups of a launch (>= 13 blocks per SM on 148 SMs)

__host__ __device__ inline int stage_of(int64_t panel) { return panel % kStage == 0 ? kStage : 128; }

template <int BITS, int KC>
__global__ void __launch_bounds__(kScoreThreads) model_score_kernel(const uint8_t* __restrict__ x, int64_t nv,
                                                                    int64_t panel, int m,
                                                                    const int32_t* __restrict__ mrows,
                                                                    const double* __restrict__ Lm,
                                                                    const int32_t* __restrict__ nm, int k, int c0,
                                                                    int64_t stages, int64_t per_range,
                                                                    double* __restrict__ part, long long* __restrict__ rpart) {
    __shared__ double Ls[kStage * KC];
    __shared__ int32_t ns[kStage];
    const int p = blockIdx.y * kScoreThreads + threadIdx.x;
    const int kc = min(KC, k - c0);
    const int sv = stage_of(panel);
    const int64_t spp = (panel + sv - 1) / sv;   // stages per panel
    double acc[KC];
#pragma unroll
    for (int c = 0; c < KC; ++c) acc[c] = 0.0;
    long long r = 0;
    const int64_t s_lo = (int64_t)blockIdx.x * per_range, s_hi = min(stages, s_lo + per_range);
    for (int64_t s = s_lo; s < s_hi; ++s) {
        const int64_t pnl = s / spp;
        const int64_t vs = pnl * panel + (s - pnl * spp) * sv;
        const int w = (int)(min(min(vs + sv, (pnl + 1) * panel), nv) - vs);
        __syncthreads();   // the previous stage is consumed
        for (int i = threadIdx.x; i < sv; i += kScoreThreads) {
            const int mr = i < w ? __ldg(mrows + vs + i) : -1;
#pragma unroll
            for (int c = 0; c < KC; ++c) Ls[i * KC + c] = (mr >= 0 && c < kc) ? __ldg(Lm + (size_t)mr * k + c0 + c) : 0.0;
            ns[i] = mr >= 0 ? __ldg(nm + mr) : 0;
        }
        __syncthreads();
        if (p >= m) continue;
        // cells after nv in the last panel are zero, and the staged rows after w are zero: whole 16-cell groups are safe
        const int64_t base = pnl * (int64_t)m * panel + (int64_t)p * panel + (vs - pnl * panel);
        for (int i = 0; i < w; i += 16) {
            int xv[16];
            load16<BITS>(x, base + i, xv);
            int any = 0;
#pragma unroll
            for (int j = 0; j < 16; ++j) any |= xv[j];
            if (any == 0) continue;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const double xd = (double)xv[j];
#pragma unroll
                for (int c = 0; c < KC; ++c) acc[c] = __fma_rn(xd, Ls[(i + j) * KC + c], acc[c]);
                r += (long long)xv[j] * ns[i + j];
            }
        }
    }
    if (p >= m) return;
#pragma unroll
    for (int c = 0; c < KC; ++c)
        if (c < kc) part[((size_t)blockIdx.x * m + p) * k + c0 + c] = acc[c];
    if (c0 == 0) rpart[(size_t)blockIdx.x * m + p] = r;
}

// acc (m x k doubles, then m int64) += sum over ranges q in ascending order of the partials
__global__ void model_fold_kernel(const double* __restrict__ part, const long long* __restrict__ rpart, int64_t ranges,
                                  int m, int k, double* __restrict__ acc) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m * (k + 1)) return;
    if (t < m * k) {
        double s = 0.0;
        for (int64_t q = 0; q < ranges; ++q) s = __dadd_rn(s, part[(size_t)q * m * k + t]);
        acc[t] = __dadd_rn(acc[t], s);
    } else {
        const int p = t - m * k;
        long long s = 0;
        for (int64_t q = 0; q < ranges; ++q) s += rpart[(size_t)q * m + p];
        reinterpret_cast<long long*>(acc + (size_t)m * k)[p] += s;
    }
}

__global__ void model_add_kernel(double* __restrict__ dst, const double* __restrict__ src, int m, int k) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < m * k) dst[t] = __dadd_rn(dst[t], src[t]);
    else if (t < m * (k + 1))
        reinterpret_cast<long long*>(dst + (size_t)m * k)[t - m * k] +=
            reinterpret_cast<const long long*>(src + (size_t)m * k)[t - m * k];
}

// a_c = sum_f u_fc, b_c = sum_f (rs_f / N) u_fc: one warp per column, ascending f per lane, then a fixed xor tree
__global__ void model_terms_kernel(const double* __restrict__ U, const double* __restrict__ rowsum, int n, int k,
                                   double* __restrict__ a, double* __restrict__ b) {
    const int c = blockIdx.x, lane = threadIdx.x;
    const double* u = U + (size_t)c * n;
    double sa = 0.0, sb = 0.0;
    for (int f = lane; f < n; f += 32) {
        sa = __dadd_rn(sa, u[f]);
        sb = __fma_rn(__ddiv_rn(rowsum[f], (double)n), u[f], sb);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sa = __dadd_rn(sa, __shfl_xor_sync(0xffffffffu, sa, o));
        sb = __dadd_rn(sb, __shfl_xor_sync(0xffffffffu, sb, o));
    }
    if (lane == 0) {
        a[c] = sa;
        b[c] = sb;
    }
}

// y[p + c m] = (((T_pc - (r_p / N) a_c) - b_c) + mean a_c) / lambda_c, in exactly this operation order
__global__ void model_finish_kernel(const double* __restrict__ acc, int m, int k, int kout, int n_fit,
                                    const double* __restrict__ terms, double* __restrict__ y) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m * kout) return;
    const int p = t / kout, c = t - p * kout;
    const double* lam = terms;
    const double* a = terms + k;
    const double* b = terms + 2 * k;
    const double mean = terms[3 * k];
    const long long r = reinterpret_cast<const long long*>(acc + (size_t)m * k)[p];
    const double rm = __ddiv_rn((double)r, (double)n_fit);
    const double v = __dadd_rn(__dsub_rn(__dsub_rn(acc[(size_t)p * k + c], __dmul_rn(rm, a[c])), b[c]), __dmul_rn(mean, a[c]));
    y[p + (size_t)c * m] = __ddiv_rn(v, lam[c]);
}

template <int KC>
cudaError_t score_launch(const uint8_t* x, int elem_bits, int64_t nv, int64_t panel, int m, const int32_t* d_mrows,
                         const double* d_L, const int32_t* d_n, int k, int64_t stages, int64_t ranges, int64_t per_range,
                         double* d_part, long long* d_rpart, cudaStream_t stream) {
    const dim3 grid((unsigned)ranges, (unsigned)((m + kScoreThreads - 1) / kScoreThreads));
    for (int c0 = 0; c0 < k; c0 += KC) {
        if (elem_bits == 8)
            model_score_kernel<8, KC><<<grid, kScoreThreads, 0, stream>>>(x, nv, panel, m, d_mrows, d_L, d_n, k, c0, stages,
                                                                          per_range, d_part, d_rpart);
        else if (elem_bits == 16)
            model_score_kernel<16, KC><<<grid, kScoreThreads, 0, stream>>>(x, nv, panel, m, d_mrows, d_L, d_n, k, c0, stages,
                                                                           per_range, d_part, d_rpart);
        else
            model_score_kernel<4, KC><<<grid, kScoreThreads, 0, stream>>>(x, nv, panel, m, d_mrows, d_L, d_n, k, c0, stages,
                                                                          per_range, d_part, d_rpart);
    }
    return cudaGetLastError();
}

void score_shape(int64_t nv, int64_t panel, int m, int64_t* stages, int64_t* ranges, int64_t* per_range) {
    const int sv = stage_of(panel);
    const int64_t spp = (panel + sv - 1) / sv;
    const int64_t full = nv / panel, rest = nv - full * panel;
    *stages = full * spp + (rest + sv - 1) / sv;
    const int64_t groups = (m + kScoreThreads - 1) / kScoreThreads;
    const int64_t want = std::max<int64_t>(1, (kMaxRangeBlocks + groups - 1) / groups);
    *per_range = std::max<int64_t>(1, (*stages + want - 1) / want);
    *ranges = (*stages + *per_range - 1) / *per_range;
}

}  // namespace

cudaError_t model_loadings(const void* d_x, int elem_bits, int64_t nv, int64_t panel, int rows, int n_fit, const double* d_u,
                           int k, double* d_L, int32_t* d_carriers, cudaStream_t stream) {
    if (nv <= 0) return cudaSuccess;
    if (k <= 2) return loadings_launch<2>(d_x, elem_bits, nv, panel, rows, n_fit, d_u, k, d_L, d_carriers, stream);
    if (k <= 4) return loadings_launch<4>(d_x, elem_bits, nv, panel, rows, n_fit, d_u, k, d_L, d_carriers, stream);
    return loadings_launch<8>(d_x, elem_bits, nv, panel, rows, n_fit, d_u, k, d_L, d_carriers, stream);
}

size_t model_score_scratch(int m, int k) {
    const int64_t groups = (m + kScoreThreads - 1) / kScoreThreads;
    const int64_t ranges = std::max<int64_t>(1, (kMaxRangeBlocks + groups - 1) / groups);
    return (size_t)ranges * m * (k + 1) * sizeof(double);
}

cudaError_t model_score(const void* d_x, int elem_bits, int64_t nv, int64_t panel, int m, const int32_t* d_mrows,
                        const double* d_L, const int32_t* d_n, int k, double* d_scratch, double* d_acc, cudaStream_t stream) {
    if (nv <= 0) return cudaSuccess;
    int64_t stages, ranges, per_range;
    score_shape(nv, panel, m, &stages, &ranges, &per_range);
    double* d_part = d_scratch;
    long long* d_rpart = reinterpret_cast<long long*>(d_scratch + (size_t)ranges * m * k);
    const uint8_t* x = static_cast<const uint8_t*>(d_x);
    cudaError_t e;
    if (k <= 2) e = score_launch<2>(x, elem_bits, nv, panel, m, d_mrows, d_L, d_n, k, stages, ranges, per_range, d_part, d_rpart, stream);
    else if (k <= 4) e = score_launch<4>(x, elem_bits, nv, panel, m, d_mrows, d_L, d_n, k, stages, ranges, per_range, d_part, d_rpart, stream);
    else e = score_launch<8>(x, elem_bits, nv, panel, m, d_mrows, d_L, d_n, k, stages, ranges, per_range, d_part, d_rpart, stream);
    if (e != cudaSuccess) return e;
    const int cells = m * (k + 1);
    model_fold_kernel<<<(cells + 255) / 256, 256, 0, stream>>>(d_part, d_rpart, ranges, m, k, d_acc);
    return cudaGetLastError();
}

cudaError_t model_terms(const double* d_u, const double* d_rowsum, int n, int k, double* d_a, double* d_b, cudaStream_t stream) {
    model_terms_kernel<<<k, 32, 0, stream>>>(d_u, d_rowsum, n, k, d_a, d_b);
    return cudaGetLastError();
}

cudaError_t model_add(double* d_dst, const double* d_src, int m, int k, cudaStream_t stream) {
    const int cells = m * (k + 1);
    model_add_kernel<<<(cells + 255) / 256, 256, 0, stream>>>(d_dst, d_src, m, k);
    return cudaGetLastError();
}

cudaError_t model_finish(const double* d_acc, int m, int k, int kout, int n_fit, const double* d_terms, double* d_y,
                         cudaStream_t stream) {
    const int cells = m * kout;
    model_finish_kernel<<<(cells + 255) / 256, 256, 0, stream>>>(d_acc, m, k, kout, n_fit, d_terms, d_y);
    return cudaGetLastError();
}

}  // namespace vpca

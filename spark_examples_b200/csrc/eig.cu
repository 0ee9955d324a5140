// Centering + symmetric eigensolve (top-k) in FP64 on the device.
//
// Replaces VariantsPcaDriver.computePca (reference:
//   src/main/scala/com/google/cloud/genomics/spark/examples/VariantsPca.scala:198-231):
//   :199-223  row sums, matrixMean = sum / N / N, C(i,j) = S(i,j) - rowMean(i) - colMean(j) + matrixMean
//   :224-227  RowMatrix(rows).computePrincipalComponents(numPc): spark-mllib 1.6.1 forms Cov = C^T C/(m-1) - ... and
//             takes the first k left singular vectors of Cov (LAPACK dgesdd).  C = J S J is symmetric PSD, so those
//             are the eigenvectors of C for its k largest eigenvalues; we compute them from C directly:
//   N >= 512 (default): Lanczos with full reorthogonalisation for the top k pairs only -- as ONE persistent cooperative
//               kernel per 16-step chunk that reads the int32 Gram S itself and applies the centring to the vector
//               (lz_persist_kernel below); the five-kernel CUDA-graph form of round 1 remains for N > 16384;
//   small N, VPCA_EIG=direct, and the fallback of the Krylov solver:
//               1. Householder tridiagonalisation  C = Q T Q^T           (N steps, 1-2 kernels per step, not blocked)
//               2. k largest eigenvalues of T by Sturm-count multisection (parallel over shifts)
//               3. eigenvectors of T by inverse iteration               (tridiagonal LU with partial pivoting)
//               4. back-transformation  z = Q y  with the stored reflectors, normalise, fix the sign.
// Everything is latency-bound FP64 vector work (at N = 2504 the matrix lives in L2, or for Lanczos in shared memory): rows
// are contiguous so every pass is coalesced.
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cstdlib>
#include <cmath>
#include <cstdint>

#include "vpca_internal.h"

namespace vpca {
namespace {

constexpr int kSmallThreads = 1024;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sum over the block; result valid in every thread.  `red` has >= 33 doubles.
__device__ __forceinline__ double block_sum(double v, double* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();   // protect `red` from the previous use
    if (lane == 0) red[wid] = v;
    __syncthreads();
    double t = (lane < nw) ? red[lane] : 0.0;
    t = warp_sum(t);
    return t;
}

// ------------------------------------------------------------------------------------------ centering
__global__ void rowsum_kernel(const int32_t* __restrict__ S, int n, double* __restrict__ rowsum) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    const int32_t* r = S + (size_t)row * n;
    long long acc = 0;
    for (int j = lane; j < n; j += 32) acc += r[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    // integer-valued and < 2^53: identical to the reference's foldLeft(0D)(_ + _) at :206
    if (lane == 0) rowsum[row] = (double)acc;
}

// scal[0] = *mm = matrixMean (:211), nz = rowSums.filter(_ > 0).size (:207).  The solvers reuse scal as scratch; *mm is
// what the projection of new rows reads.
__global__ void matrix_mean_kernel(const double* __restrict__ rowsum, int n, double* __restrict__ scal,
                                   int* __restrict__ nz, double* __restrict__ mm) {
    __shared__ double red[33];
    __shared__ int cnt;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    double acc = 0.0;
    int c = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double r = rowsum[i];
        acc += r;   // exact: integer-valued partial sums below 2^53, so the order of `reduce(_ + _)` (:210) is immaterial
        c += (r > 0.0);
    }
    const double tot = block_sum(acc, red);
    atomicAdd(&cnt, c);
    __syncthreads();
    if (threadIdx.x == 0) {
        const double rc = (double)n;
        scal[0] = __ddiv_rn(__ddiv_rn(tot, rc), rc);
        *mm = scal[0];
        *nz = cnt;
    }
}

__global__ void center_kernel(const int32_t* __restrict__ S, const double* __restrict__ rowsum,
                              const double* __restrict__ scal, int n, double* __restrict__ C) {
    const int row = blockIdx.y;
    const double rc = (double)n;
    const double row_mean = __ddiv_rn(rowsum[row], rc);
    const double mm = scal[0];
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const double col_mean = __ddiv_rn(rowsum[j], rc);
        const double data = (double)S[(size_t)row * n + j];
        // data - rowMean - colMean + matrixMean, left to right (:221)
        C[(size_t)row * n + j] = __dadd_rn(__dsub_rn(__dsub_rn(data, row_mean), col_mean), mm);
    }
}

// ---------------------------------------------------------------------------- tridiagonalisation
// Step j (0 <= j <= n-1), single block:
//   (a) finish the previous step: w = p - (tau_prev/2)(p.v_prev) v_prev          on indices [j, n)
//   (b) apply the pending rank-2 update to row j:  A[j][t] -= v_prev[j] w[t] + w[j] v_prev[t],  t in [j, n)
//   (c) d[j] = A[j][j];  build the reflector that annihilates A[j][j+2..n):  v (v[j+1] = 1), tau, e[j] = beta;
//       the reflector is kept in row j of A (for the back-transformation) and in `vcur`.
// vprev/vcur/w/p are length-n vectors; scal[1] = tau_prev on entry, tau_j on exit.
// The step index j lives in device memory (step[0] = next step, step[1] = step of the pending big kernel) so that
// every launch of the step loop is identical and the loop can be replayed from one CUDA graph.
__global__ void __launch_bounds__(kSmallThreads) tridiag_small_kernel(double* __restrict__ A, int n,
                                                                       int* __restrict__ step, double* __restrict__ v2,
                                                                       const double* __restrict__ p,
                                                                       double* __restrict__ w, double* __restrict__ diag,
                                                                       double* __restrict__ off, double* __restrict__ tau,
                                                                       double* __restrict__ scal) {
    __shared__ double red[33];
    __shared__ double bcast[2];
    const int tid = threadIdx.x, nt = blockDim.x;
    const int j = step[0];
    if (j >= n) return;
    const double* vprev = v2 + (size_t)((j + 1) & 1) * n;
    double* vcur = v2 + (size_t)(j & 1) * n;
    double* rowj = A + (size_t)j * n;
    double acc = 0.0;
    if (j > 0) {
        // (a) + (b) in two passes: the dot product, then w and the updated row together (w[j] is recomputed locally)
        const double tau_prev = tau[j - 1];
        for (int t = j + tid; t < n; t += nt) acc += p[t] * vprev[t];
        const double alpha = 0.5 * tau_prev * block_sum(acc, red);
        const double vj = vprev[j];
        const double wj = p[j] - alpha * vj;
        acc = 0.0;
        for (int t = j + tid; t < n; t += nt) {
            const double vt = vprev[t];
            const double wt = p[t] - alpha * vt;
            w[t] = wt;
            const double r = rowj[t] - (vj * wt + wj * vt);
            rowj[t] = r;
            if (t >= j + 2) acc += r * r;
            if (t == j) bcast[0] = r;
            if (t == j + 1) bcast[1] = r;
        }
    } else {
        for (int t = tid; t < n; t += nt) {
            const double r = rowj[t];
            if (t >= 2) acc += r * r;
            if (t == 0) bcast[0] = r;
            if (t == 1) bcast[1] = r;
        }
    }
    const double xnorm2 = block_sum(acc, red);     // its barriers also publish bcast[]
    if (tid == 0) diag[j] = bcast[0];
    if (j >= n - 1) {
        if (tid == 0) {
            step[1] = j;
            step[0] = j + 1;
        }
        return;
    }
    // (c) reflector from x = rowj[j+1 .. n)
    const double alpha1 = bcast[1];
    double beta, tj, scale;
    if (xnorm2 == 0.0) {
        beta = alpha1;
        tj = 0.0;
        scale = 0.0;
    } else {
        beta = -copysign(sqrt(alpha1 * alpha1 + xnorm2), alpha1);
        tj = (beta - alpha1) / beta;
        scale = 1.0 / (alpha1 - beta);
    }
    for (int t = j + 1 + tid; t < n; t += nt) {
        const double v = (t == j + 1) ? 1.0 : rowj[t] * scale;
        vcur[t] = v;
        rowj[t] = v;
    }
    if (tid == 0) {
        off[j] = beta;
        tau[j] = tj;
        scal[1] = tj;
        step[1] = j;
        step[0] = j + 1;
    }
}

// Step j, grid-wide: for every trailing row i in [j+1, n) (one warp per row, 4 rows per block)
//   A[i][t] -= vprev[i] w[t] + w[i] vprev[t]      (pending rank-2 update of step j-1),  t in [j+1, n)
//   p[i]     = tau_j * sum_t A[i][t] vcur[t]      (symmetric matrix-vector product of step j, full rows)
// The loop is unrolled by 4 so that every lane keeps four independent 8-byte loads of the (L2-resident) matrix in
// flight; the three vectors are L1 hits.
__global__ void __launch_bounds__(128) tridiag_big_kernel(double* __restrict__ A, int n, const int* __restrict__ step,
                                                          const double* __restrict__ v2,
                                                          const double* __restrict__ w, const double* __restrict__ tau,
                                                          double* __restrict__ p) {
    const int lane = threadIdx.x & 31;
    const int j = step[1];
    const int i = j + 1 + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= n) return;
    const double* __restrict__ vprev = v2 + (size_t)((j + 1) & 1) * n;
    const double* __restrict__ vcur = v2 + (size_t)(j & 1) * n;
    const double tj = tau[j];
    double* row = A + (size_t)i * n;
    const double vi = vprev[i], wi = w[i];
    double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
    int t = j + 1 + lane;
    if (j > 0) {
        for (; t + 96 < n; t += 128) {
            const double r0 = row[t], r1 = row[t + 32], r2 = row[t + 64], r3 = row[t + 96];
            const double a0 = r0 - (vi * w[t] + wi * vprev[t]);
            const double a1 = r1 - (vi * w[t + 32] + wi * vprev[t + 32]);
            const double a2 = r2 - (vi * w[t + 64] + wi * vprev[t + 64]);
            const double a3 = r3 - (vi * w[t + 96] + wi * vprev[t + 96]);
            row[t] = a0; row[t + 32] = a1; row[t + 64] = a2; row[t + 96] = a3;
            acc0 += a0 * vcur[t]; acc1 += a1 * vcur[t + 32]; acc2 += a2 * vcur[t + 64]; acc3 += a3 * vcur[t + 96];
        }
        for (; t < n; t += 32) {
            const double a = row[t] - (vi * w[t] + wi * vprev[t]);
            row[t] = a;
            acc0 += a * vcur[t];
        }
    } else {
        for (; t + 96 < n; t += 128) {
            acc0 += row[t] * vcur[t]; acc1 += row[t + 32] * vcur[t + 32];
            acc2 += row[t + 64] * vcur[t + 64]; acc3 += row[t + 96] * vcur[t + 96];
        }
        for (; t < n; t += 32) acc0 += row[t] * vcur[t];
    }
    const double acc = warp_sum((acc0 + acc1) + (acc2 + acc3));
    if (lane == 0) p[i] = tj * acc;
}

// One launch per Householder step (used when 3 n doubles fit in shared memory).  Every block redundantly redoes the
// O(n) serial part of the step in its own shared memory -- w of the previous step, the updated row j, reflector j --
// and then applies the pending rank-2 update to ITS rows fused with the mat-vec of step j.  No single-block kernel
// sits on the critical path any more; the redundant vector reads are ~10 % of the matrix traffic at 1 block per SM.
//   p2 : two length-n buffers, step j reads p_{j-1} from p2[(j+1)&1] and writes p_j to p2[j&1]
//   v2 : two length-n buffers, block 0 publishes v_j in v2[j&1]; v_{j-1} is read from v2[(j+1)&1]
// Reflector j-1 is copied into row j-1 of A by block 0 of step j (row j-1 has no readers any more by then).
__global__ void __launch_bounds__(512) tridiag_fused_kernel(double* __restrict__ A, int n, int* __restrict__ step,
                                                            double* __restrict__ v2, double* __restrict__ p2,
                                                            double* __restrict__ diag, double* __restrict__ off,
                                                            double* __restrict__ tau) {
    extern __shared__ double fsm[];
    __shared__ double red[33];
    __shared__ double bc[2];
    __shared__ int is_last;
    double* vp = fsm;             // v_{j-1}
    double* w = fsm + n;          // w_{j-1}
    double* v = fsm + 2 * (size_t)n;   // row j after the pending update, then v_j
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31;
    const int j = step[1];
    if (j >= n) return;
    const double* vprev_g = v2 + (size_t)((j + 1) & 1) * n;
    const double* p_in = p2 + (size_t)((j + 1) & 1) * n;
    double* p_out = p2 + (size_t)(j & 1) * n;
    double* rowj = A + (size_t)j * n;
    // ---- serial part, redundantly per block
    double acc = 0.0;
    if (j > 0) {
        for (int t = j + tid; t < n; t += nt) {
            const double a = vprev_g[t], b = p_in[t];
            vp[t] = a;
            w[t] = b;                      // p for now
            acc += a * b;
        }
    }
    const double pv = block_sum(acc, red);                       // (barriers also publish vp / w)
    const double alpha = (j > 0) ? 0.5 * tau[j - 1] * pv : 0.0;
    const double vj = (j > 0) ? vp[j] : 0.0;
    const double wj = (j > 0) ? w[j] - alpha * vj : 0.0;
    __syncthreads();                                             // everyone has read w[j] before it is overwritten
    acc = 0.0;
    for (int t = j + tid; t < n; t += nt) {
        double r = rowj[t];
        if (j > 0) {
            const double vt = vp[t];
            const double wt = w[t] - alpha * vt;
            w[t] = wt;
            r -= vj * wt + wj * vt;
        } else {
            vp[t] = 0.0;
            w[t] = 0.0;
        }
        v[t] = r;
        if (t >= j + 2) acc += r * r;
        if (t == j) bc[0] = r;
        if (t == j + 1) bc[1] = r;
    }
    const double xnorm2 = block_sum(acc, red);
    double beta = 0.0, tj = 0.0, scale = 0.0;
    if (j < n - 1) {
        const double a1 = bc[1];
        if (xnorm2 == 0.0) {
            beta = a1;
        } else {
            beta = -copysign(sqrt(a1 * a1 + xnorm2), a1);
            tj = (beta - a1) / beta;
            scale = 1.0 / (a1 - beta);
        }
        for (int t = j + 1 + tid; t < n; t += nt) v[t] = (t == j + 1) ? 1.0 : v[t] * scale;
    }
    __syncthreads();
    if (blockIdx.x == 0) {
        if (tid == 0) {
            diag[j] = bc[0];
            if (j < n - 1) {
                off[j] = beta;
                tau[j] = tj;
            }
        }
        double* vout = v2 + (size_t)(j & 1) * n;
        for (int t = j + 1 + tid; t < n; t += nt) vout[t] = v[t];
        if (j > 0) {
            double* store = A + (size_t)(j - 1) * n;             // reflector j-1 for the back-transformation
            for (int t = j + tid; t < n; t += nt) store[t] = vp[t];
        }
    }
    // ---- this block's share of the trailing rows: pending update fused with the mat-vec of step j
    if (j < n - 1) {
        const int warps = nt >> 5;
        for (int i = j + 1 + blockIdx.x * warps + (tid >> 5); i < n; i += gridDim.x * warps) {
            double* row = A + (size_t)i * n;
            const double vi = vp[i], wi = w[i];
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            int t = j + 1 + lane;
            if (j > 0) {
                // 4 independent 8-byte loads per lane in flight (8 was measured slower: 53 vs 42.5 ms at N = 2504)
                for (; t + 96 < n; t += 128) {
                    const double r0 = row[t], r1 = row[t + 32], r2 = row[t + 64], r3 = row[t + 96];
                    const double u0 = r0 - (vi * w[t] + wi * vp[t]);
                    const double u1 = r1 - (vi * w[t + 32] + wi * vp[t + 32]);
                    const double u2 = r2 - (vi * w[t + 64] + wi * vp[t + 64]);
                    const double u3 = r3 - (vi * w[t + 96] + wi * vp[t + 96]);
                    row[t] = u0; row[t + 32] = u1; row[t + 64] = u2; row[t + 96] = u3;
                    a0 += u0 * v[t]; a1 += u1 * v[t + 32]; a2 += u2 * v[t + 64]; a3 += u3 * v[t + 96];
                }
                for (; t < n; t += 32) {
                    const double u = row[t] - (vi * w[t] + wi * vp[t]);
                    row[t] = u;
                    a0 += u * v[t];
                }
            } else {
                for (; t + 96 < n; t += 128) {
                    a0 += row[t] * v[t]; a1 += row[t + 32] * v[t + 32];
                    a2 += row[t + 64] * v[t + 64]; a3 += row[t + 96] * v[t + 96];
                }
                for (; t < n; t += 32) a0 += row[t] * v[t];
            }
            const double sum = warp_sum((a0 + a1) + (a2 + a3));
            if (lane == 0) p_out[i] = tj * sum;
        }
    }
    // ---- the last block to finish advances the step (every block has read it by then)
    __threadfence();
    __syncthreads();
    if (tid == 0) is_last = (atomicAdd(step + 2, 1) == (int)gridDim.x - 1);
    __syncthreads();
    if (is_last && tid == 0) {
        step[2] = 0;
        step[1] = j + 1;
    }
}

// ------------------------------------------------------------------------- eigenvalues of T (bisection)
// Number of eigenvalues of T strictly below x (Sturm count with the LAPACK dlaebz pivmin safeguard).
__device__ __forceinline__ int sturm_count(const double* __restrict__ d, const double* __restrict__ e2, int n,
                                           double x, double pivmin) {
    double q = d[0] - x;
    if (fabs(q) < pivmin) q = -pivmin;
    int cnt = q < 0.0;
    for (int i = 1; i < n; ++i) {
        q = d[i] - x - e2[i - 1] / q;
        if (fabs(q) < pivmin) q = -pivmin;
        cnt += q < 0.0;
    }
    return cnt;
}

// block b computes the (b+1)-th largest eigenvalue by multisection: every round each thread counts at one shift.
__global__ void __launch_bounds__(256) bisect_kernel(const double* __restrict__ d, const double* __restrict__ e, int n,
                                                     double* __restrict__ e2, double* __restrict__ evals,
                                                     double* __restrict__ scal, const int* __restrict__ gate = nullptr) {
    __shared__ int sel;
    __shared__ double sh_lo, sh_hi, sh_piv;
    if (gate != nullptr && *gate == 0) return;   // speculatively enqueued behind a convergence test that failed
    const int tid = threadIdx.x, nt = blockDim.x;
    // Gershgorin interval, pivmin, squared off-diagonals (every block writes the same e2 values)
    double gl = DBL_MAX, gu = -DBL_MAX, emax = 0.0;
    for (int i = tid; i < n; i += nt) {
        const double el = (i > 0) ? fabs(e[i - 1]) : 0.0, er = (i < n - 1) ? fabs(e[i]) : 0.0;
        gl = fmin(gl, d[i] - el - er);
        gu = fmax(gu, d[i] + el + er);
        if (i < n - 1) {
            e2[i] = e[i] * e[i];
            emax = fmax(emax, e[i] * e[i]);
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        gl = fmin(gl, __shfl_xor_sync(0xffffffffu, gl, o));
        gu = fmax(gu, __shfl_xor_sync(0xffffffffu, gu, o));
        emax = fmax(emax, __shfl_xor_sync(0xffffffffu, emax, o));
    }
    __shared__ double rl[8], ru[8], rm[8];
    if ((tid & 31) == 0) {
        rl[tid >> 5] = gl;
        ru[tid >> 5] = gu;
        rm[tid >> 5] = emax;
    }
    __syncthreads();
    if (tid == 0) {
        double a = rl[0], b = ru[0], m = rm[0];
        for (int i = 1; i < (nt >> 5); ++i) {
            a = fmin(a, rl[i]);
            b = fmax(b, ru[i]);
            m = fmax(m, rm[i]);
        }
        const double tnorm = fmax(fabs(a), fabs(b));
        sh_piv = DBL_MIN * fmax(1.0, m);
        sh_lo = a - 2.0 * tnorm * DBL_EPSILON * n - 2.0 * sh_piv;
        sh_hi = b + 2.0 * tnorm * DBL_EPSILON * n + 2.0 * sh_piv;
        if (blockIdx.x == 0) scal[2] = tnorm;
    }
    __syncthreads();
    const double pivmin = sh_piv;
    const int target = n - 1 - (int)blockIdx.x;   // ascending index of the wanted eigenvalue
    double lo = sh_lo, hi = sh_hi;                // invariant: count(lo) <= target < count(hi)
    for (int round = 0; round < 16; ++round) {
        const double width = hi - lo;
        if (width <= 2.0 * DBL_EPSILON * fmax(fabs(lo), fabs(hi)) + 2.0 * pivmin) break;
        const double x = lo + width * ((double)(tid + 1) / (double)(nt + 1));
        const int c = sturm_count(d, e2, n, x, pivmin);
        if (tid == 0) sel = nt;
        __syncthreads();
        if (c > target) atomicMin(&sel, tid);   // first shift with more than `target` eigenvalues below it
        __syncthreads();
        const int s = sel;
        const double nlo = (s == 0) ? lo : lo + width * ((double)s / (double)(nt + 1));
        const double nhi = (s == nt) ? hi : lo + width * ((double)(s + 1) / (double)(nt + 1));
        __syncthreads();
        lo = nlo;
        hi = nhi;
    }
    if (tid == 0) evals[blockIdx.x] = 0.5 * (lo + hi);
}

// ------------------------------------------------------------- eigenvectors of T (inverse iteration)
__device__ __forceinline__ double block_max(double v, double* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    double t = (lane < nw) ? red[lane] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t = fmax(t, __shfl_xor_sync(0xffffffffu, t, o));
    return t;
}

// One block; the k eigenvalues are processed one after the other.  The tridiagonal LU (partial pivoting) and the
// two substitutions are serial recurrences run by thread 0 out of shared memory (SMEM) or an 8n-double global
// scratch; dot products / scaling run on the whole block.  Y: n x k column-major, unit 2-norm eigenvectors of T.
template <bool SMEM>
__global__ void __launch_bounds__(256) invit_kernel(const double* __restrict__ d, const double* __restrict__ e, int n,
                                                    int k, const double* __restrict__ evals,
                                                    const double* __restrict__ scal, double* __restrict__ scratch,
                                                    double* __restrict__ Y) {
    extern __shared__ double sm[];
    __shared__ double red[33];
    double* base = SMEM ? sm : scratch;
    double* sd = base;
    double* se = base + (size_t)n;
    double* u0 = base + 2 * (size_t)n;
    double* u1 = base + 3 * (size_t)n;
    double* u2 = base + 4 * (size_t)n;
    double* lm = base + 5 * (size_t)n;
    double* pv = base + 6 * (size_t)n;
    double* y = base + 7 * (size_t)n;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int i = tid; i < n; i += nt) {
        sd[i] = d[i];
        se[i] = (i < n - 1) ? e[i] : 0.0;
    }
    __syncthreads();
    const double tnorm = fmax(scal[2], DBL_MIN);
    const double tiny = DBL_EPSILON * tnorm;
    for (int c = 0; c < k; ++c) {
        if (tid == 0) {
            double lam = evals[c];
            // separate numerically coincident eigenvalues a little (LAPACK dstein does the same)
            if (c > 0 && fabs(lam - evals[c - 1]) < 10.0 * tiny) lam = evals[c - 1] - 10.0 * tiny;
            // factor T - lam I = P L U, U with two super-diagonals
            double cur_d = sd[0] - lam, cur_u = (n > 1) ? se[0] : 0.0;
            for (int i = 0; i < n - 1; ++i) {
                const double sub = se[i];
                const double next_d = sd[i + 1] - lam;
                const double next_u = (i + 1 < n - 1) ? se[i + 1] : 0.0;
                if (fabs(cur_d) >= fabs(sub)) {
                    if (fabs(cur_d) < tiny) cur_d = copysign(tiny, cur_d);
                    const double m = sub / cur_d;
                    lm[i] = m;
                    pv[i] = 0.0;
                    u0[i] = cur_d;
                    u1[i] = cur_u;
                    u2[i] = 0.0;
                    cur_d = next_d - m * cur_u;
                    cur_u = next_u;
                } else {
                    const double m = cur_d / sub;
                    lm[i] = m;
                    pv[i] = 1.0;
                    u0[i] = sub;
                    u1[i] = next_d;
                    u2[i] = next_u;
                    cur_d = cur_u - m * next_d;
                    cur_u = -m * next_u;
                }
            }
            if (fabs(cur_d) < tiny) cur_d = copysign(tiny, cur_d);
            u0[n - 1] = cur_d;
            u1[n - 1] = 0.0;
            u2[n - 1] = 0.0;
        }
        for (int i = tid; i < n; i += nt) y[i] = 1.0;
        for (int itn = 0; itn < 4; ++itn) {
            __syncthreads();
            if (tid == 0) {
                if (itn > 0) {   // forward substitution with the row interchanges (skipped on the first pass)
                    for (int i = 0; i < n - 1; ++i) {
                        if (pv[i] != 0.0) {
                            const double t = y[i];
                            y[i] = y[i + 1];
                            y[i + 1] = t;
                        }
                        y[i + 1] -= lm[i] * y[i];
                    }
                }
                y[n - 1] = y[n - 1] / u0[n - 1];
                if (n > 1) y[n - 2] = (y[n - 2] - u1[n - 2] * y[n - 1]) / u0[n - 2];
                for (int i = n - 3; i >= 0; --i) y[i] = (y[i] - u1[i] * y[i + 1] - u2[i] * y[i + 2]) / u0[i];
            }
            __syncthreads();
            // scale to unit max-norm first (the solve may have grown the vector by 1/eps), then orthogonalise
            double mx = 0.0;
            for (int i = tid; i < n; i += nt) mx = fmax(mx, fabs(y[i]));
            mx = block_max(mx, red);
            const double inv = 1.0 / fmax(mx, DBL_MIN);
            for (int i = tid; i < n; i += nt) y[i] *= inv;
            for (int q = 0; q < c; ++q) {
                const double* z = Y + (size_t)q * n;
                double acc = 0.0;
                for (int i = tid; i < n; i += nt) acc += z[i] * y[i];
                const double dot = block_sum(acc, red);
                for (int i = tid; i < n; i += nt) y[i] -= dot * z[i];
            }
        }
        __syncthreads();
        double acc = 0.0;
        for (int i = tid; i < n; i += nt) acc += y[i] * y[i];
        const double inv = 1.0 / sqrt(block_sum(acc, red));
        for (int i = tid; i < n; i += nt) Y[(size_t)c * n + i] = y[i] * inv;
        __syncthreads();
    }
}

// Unit 2-norm, then the sign rule: the largest-|.| entry (lowest index on ties) is positive.  Whole block, y of length n.
__device__ void normalise_and_orient(double* __restrict__ y, int n) {
    __shared__ double red[33];
    __shared__ int arg;
    __shared__ double bv[32];
    __shared__ int bi[32];
    const int tid = threadIdx.x, nt = blockDim.x;
    double acc = 0.0;
    for (int t = tid; t < n; t += nt) acc += y[t] * y[t];
    const double inv = 1.0 / sqrt(block_sum(acc, red));
    double best = -1.0;
    int besti = n;
    for (int t = tid; t < n; t += nt) {
        const double a = fabs(y[t]);
        if (a > best) {
            best = a;
            besti = t;
        }
    }
    // block arg-max (value, then lowest index)
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
        if (ov > best || (ov == best && oi < besti)) {
            best = ov;
            besti = oi;
        }
    }
    if ((tid & 31) == 0) {
        bv[tid >> 5] = best;
        bi[tid >> 5] = besti;
    }
    __syncthreads();
    if (tid == 0) {
        double b = bv[0];
        int ix = bi[0];
        for (int i = 1; i < (nt >> 5); ++i)
            if (bv[i] > b || (bv[i] == b && bi[i] < ix)) {
                b = bv[i];
                ix = bi[i];
            }
        arg = ix;
    }
    __syncthreads();
    const double sgn = (y[arg] < 0.0) ? -inv : inv;
    __syncthreads();
    for (int t = tid; t < n; t += nt) y[t] *= sgn;
}

// ----------------------------------------------------------------------------- back-transformation
// z = H_0 H_1 ... H_{n-2} y, H_j = I - tau_j v_j v_j^T with v_j in row j of A at [j+1, n).  One block per eigenvector.
__global__ void __launch_bounds__(512) backtransform_kernel(const double* __restrict__ A, int n,
                                                            const double* __restrict__ tau, double* __restrict__ Y) {
    __shared__ double red[33];
    double* y = Y + (size_t)blockIdx.x * n;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int j = n - 2; j >= 0; --j) {
        const double tj = tau[j];
        if (tj == 0.0) continue;
        const double* v = A + (size_t)j * n;
        double acc = 0.0;
        for (int t = j + 1 + tid; t < n; t += nt) acc += v[t] * y[t];
        const double s = tj * block_sum(acc, red);
        for (int t = j + 1 + tid; t < n; t += nt) y[t] -= s * v[t];
        __syncthreads();
    }
    normalise_and_orient(y, n);
}

// ------------------------------------------------- Lanczos: the top-k eigenpairs without tridiagonalising C
// For N >= kLzMinN the k largest eigenpairs come from a Krylov space instead of the full reduction: m steps of
// symmetric Lanczos with full (twice-applied classical Gram-Schmidt) reorthogonalisation build an orthonormal
// V (N x m) and a small tridiagonal T_m = V^T C V; its top-k eigenpairs (same bisection + inverse iteration as
// above, on m instead of N) give Ritz values theta and vectors z = V y whose residual is |beta_m y_m|.  One step
// costs one pass over C (50 MB from L2 at N = 2504) instead of the N steps the reduction needs, and population
// structure separates the top of the spectrum, so a few dozen steps reach |beta_m y_m| <= 1e-12 ||T||.
// Graph form (N > 16384, VPCA_LZ_PERSIST=0): five launches per step (matvec | V^T w | w -= V h | V^T w | w -= V h), step
// index and stop flag in device memory so that kLzChunk steps replay from one CUDA graph; the host looks at the residual
// after a replay.  Persistent form (default): see lz_persist_kernel further down.
// Anything unusual -- breakdown, slow convergence, a larger eigenvalue found by the deflated re-run that guards
// against a missed copy of a multiple eigenvalue -- falls back to the direct reduction, which remains the
// reference-grade path.  Every reduction has a fixed order: the result is run-to-run deterministic.
constexpr int kLzMinN = 512;         // below this the direct reduction is as fast
constexpr int kLzForcedMinN = 96;    // VPCA_EIG=lanczos: smallest n the chunked loop supports (tests)
constexpr int kLzChunk = 16;      // steps per chunk (population structure converges the top pairs in <= 16)
constexpr int kLzVerify = 8;      // steps of the deflated re-run (persistent form): its top Ritz value only has to climb ABOVE
                                  // theta_k when a copy of a larger eigenvalue was missed, not to converge
constexpr int kLzMaxIter = 320;   // give up (-> direct solver) beyond this
constexpr int kLzCap = kLzMaxIter + 64;   // columns of V: main run, or k locked vectors + one verification chunk
// st[0] = step j, st[1] = flag (0 run, 1 converged, 2 breakdown, 3 missed eigenvalue), st[2] = ticket, st[3] = step cap

__device__ __forceinline__ double lz_uniform(unsigned long long i, unsigned long long salt) {
    unsigned long long z = (i + 1) * 0x9E3779B97F4A7C15ull + salt;   // splitmix64
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (double)(z >> 11) * (1.0 / 9007199254740992.0) - 0.5;
}

// <<<ceil(n/32), 32>>>: start vector (not yet normalised) and the per-block partial sums of its squared norm
__global__ void lz_init_kernel(double* __restrict__ w, int n, unsigned long long salt, double* __restrict__ part,
                               const int* __restrict__ gate = nullptr) {
    if (gate != nullptr && *gate == 0) return;
    const int i = blockIdx.x * 32 + threadIdx.x;
    double v = 0.0;
    if (i < n) {
        v = lz_uniform((unsigned long long)i, salt);
        w[i] = v;
    }
    const double s = warp_sum(v * v);
    if (threadIdx.x == 0) part[blockIdx.x] = s;
}

// Step j, phase 1: beta_j = ||w_in|| (from the partial sums), v_j = w_in / beta_j -> V[:, j], w_out = C v_j.
// 4 rows per 256-thread block, two warps per row, 8 independent loads in flight per lane.
__global__ void __launch_bounds__(256) lz_matvec_kernel(const double* __restrict__ C, int n, double* __restrict__ V,
                                                        double* __restrict__ wbuf, const double* __restrict__ part,
                                                        int npart, double* __restrict__ beta, int* __restrict__ st) {
    __shared__ double half[8];
    const int j = st[0];
    if (st[1] != 0 || j >= st[3]) return;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    double s = 0.0;
    for (int p = lane; p < npart; p += 32) s += part[p];
    s = warp_sum(s);
    const double nrm = sqrt(s);
    if (!(nrm > 0.0) || !(nrm <= DBL_MAX)) {   // exact breakdown or non-finite: every block sees the same value
        if (blockIdx.x == 0 && threadIdx.x == 0) st[1] = 2;
        return;
    }
    const double inv = 1.0 / nrm;
    const double* __restrict__ win = wbuf + (size_t)(j & 1) * n;
    double* __restrict__ wout = wbuf + (size_t)((j + 1) & 1) * n;
    const int row = blockIdx.x * 4 + (wid >> 1);
    double acc = 0.0;
    if (row < n) {
        const double* __restrict__ c = C + (size_t)row * n;
        double a[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        for (int t0 = (wid & 1) * 32 + lane; t0 < n; t0 += 8 * 64) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {   // predicated, so the 8 loads of the ragged last round still issue together
                const int t = t0 + u * 64;
                if (t < n) a[u] += c[t] * win[t];
            }
        }
        acc = ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]));
    }
    acc = warp_sum(acc);
    if (lane == 0) half[wid] = acc;
    __syncthreads();
    if (row < n && (wid & 1) == 0 && lane == 0) {
        wout[row] = (half[wid] + half[wid + 1]) * inv;
        V[(size_t)j * n + row] = win[row] * inv;
        if (row == 0) beta[j] = nrm;
    }
}

// Phases 2 and 4: h[q] = V[:, q] . w for q <= j.  One block per column (blocks beyond j return).
__global__ void __launch_bounds__(128) lz_dots_kernel(const double* __restrict__ V, int n,
                                                      const double* __restrict__ wbuf, double* __restrict__ h,
                                                      const int* __restrict__ st) {
    __shared__ double red[33];
    const int j = st[0];
    if (st[1] != 0 || j >= st[3]) return;
    const int q = blockIdx.x;
    if (q > j) return;
    const double* __restrict__ w = wbuf + (size_t)((j + 1) & 1) * n;
    const double* __restrict__ v = V + (size_t)q * n;
    double a[4] = {0.0, 0.0, 0.0, 0.0};
    for (int t0 = threadIdx.x; t0 < n; t0 += 4 * 128) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int t = t0 + u * 128;
            if (t < n) a[u] += v[t] * w[t];
        }
    }
    const double sum = block_sum((a[0] + a[1]) + (a[2] + a[3]), red);
    if (threadIdx.x == 0) h[q] = sum;
}

// Phases 3 and 5: w -= V[:, 0..j] h.  32 rows per block, the columns split over the 8 warps.  The second pass also
// leaves the partial sums of ||w||^2 for the next step and, through a ticket, advances the step counter once every
// block has read it.  alpha_j = h_j (first pass) + its correction (second pass).
__global__ void __launch_bounds__(256) lz_update_kernel(const double* __restrict__ V, int n, double* __restrict__ wbuf,
                                                        const double* __restrict__ h, double* __restrict__ alpha,
                                                        double* __restrict__ part, int* __restrict__ st, int pass) {
    __shared__ double sm[8][33];
    const int j = st[0];
    if (st[1] != 0 || j >= st[3]) return;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int row = blockIdx.x * 32 + lane;
    double* __restrict__ w = wbuf + (size_t)((j + 1) & 1) * n;
    double acc = 0.0;
    if (row < n) {
#pragma unroll 4
        for (int q = wid; q <= j; q += 8) acc += V[(size_t)q * n + row] * h[q];
    }
    sm[wid][lane] = acc;
    __syncthreads();
    if (wid == 0) {
        const double tot = ((sm[0][lane] + sm[1][lane]) + (sm[2][lane] + sm[3][lane])) +
                           ((sm[4][lane] + sm[5][lane]) + (sm[6][lane] + sm[7][lane]));
        double nw = 0.0;
        if (row < n) {
            nw = w[row] - tot;
            w[row] = nw;
        }
        if (pass == 2) {
            const double s2 = warp_sum(nw * nw);
            if (lane == 0) part[blockIdx.x] = s2;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) alpha[j] = (pass == 1) ? h[j] : alpha[j] + h[j];
    if (pass == 2 && threadIdx.x == 0) {
        if (atomicAdd(st + 2, 1) == (int)gridDim.x - 1) {
            st[2] = 0;
            st[0] = j + 1;
        }
    }
}

// One warp.  res[0] = max_c |beta_m Y[m-1, c]| / ||T||, res[1] = beta_m; flags convergence (or NaN -> breakdown).
__global__ void lz_check_kernel(const double* __restrict__ part, int npart, const double* __restrict__ Y, int m, int k,
                                const double* __restrict__ scal, int* __restrict__ st, double* __restrict__ res,
                                double tol) {
    const int lane = threadIdx.x;
    double s = 0.0;
    for (int p = lane; p < npart; p += 32) s += part[p];
    s = warp_sum(s);
    if (lane != 0) return;
    const double nrm = sqrt(s);
    const double tnorm = fmax(scal[2], DBL_MIN);
    double r = 0.0;
    for (int c = 0; c < k; ++c) r = fmax(r, fabs(Y[(size_t)c * m + (m - 1)]));
    const double rho = nrm * r / tnorm;
    res[0] = rho;
    res[1] = nrm;
    if (st[1] == 0) {
        if (!(rho == rho) || !(rho <= DBL_MAX)) st[1] = 2;
        else if (rho <= tol) st[1] = 1;
    }
}

// Z[:, c] = V[:, 0..m) Y[:, c]; grid (ceil(n/32), k), 32 rows per block, the columns split over the 8 warps.
__global__ void __launch_bounds__(256) lz_ritz_kernel(const double* __restrict__ V, int n, const double* __restrict__ Y,
                                                      int m, double* __restrict__ Z) {
    __shared__ double sm[8][33];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int row = blockIdx.x * 32 + lane;
    const double* __restrict__ y = Y + (size_t)blockIdx.y * m;
    double acc = 0.0;
    if (row < n) {
#pragma unroll 4
        for (int q = wid; q < m; q += 8) acc += V[(size_t)q * n + row] * y[q];
    }
    sm[wid][lane] = acc;
    __syncthreads();
    if (wid == 0 && row < n)
        Z[(size_t)blockIdx.y * n + row] = ((sm[0][lane] + sm[1][lane]) + (sm[2][lane] + sm[3][lane])) +
                                          ((sm[4][lane] + sm[5][lane]) + (sm[6][lane] + sm[7][lane]));
}

__global__ void __launch_bounds__(512) lz_finish_kernel(double* __restrict__ Z, int n, const int* __restrict__ gate = nullptr) {
    if (gate != nullptr && *gate == 0) return;
    normalise_and_orient(Z + (size_t)blockIdx.x * n, n);
}

// One thread: the deflated re-run found a Ritz value above theta_k -> an eigenvalue was missed.
__global__ void lz_verify_kernel(const double* __restrict__ theta, int k, const double* __restrict__ theta2,
                                 const double* __restrict__ scal, int* __restrict__ st, const int* __restrict__ gate = nullptr) {
    if (gate != nullptr && *gate == 0) return;
    const double tnorm = fmax(scal[2], DBL_MIN);
    if (st[1] == 2) return;
    st[1] = (theta2[0] > theta[k - 1] + 1e-9 * tnorm) ? 3 : 1;
}


// ------------------------------------------------------------------ Lanczos, persistent form (n <= kLzPersistMaxN)
// The five launches of a step (and the 80 of a 16-step chunk) become ONE cooperative launch per chunk: 1024 threads on
// every SM, block b owns the rows [b R, (b + 1) R) of everything (R = ceil(n / blocks)), and a step is three phases
// separated by grid-wide barriers (an atomic counter in L2, ~1-2 us each instead of a kernel boundary):
//   A  every block stages the whole w_in in shared memory (computing ||w_in||, sum(w_in) and rowmean . w_in on the way,
//      all in one fixed order, so every block derives the same beta_j), then its rows of  y = C v_j  -- read from the
//      int32 Gram S, not from the FP64 centred matrix: (C v)_i = (S v)_i - rbar_i sum(v) - rbar . v + mean sum(v) with
//      rbar = rowSums / N (VariantsPca.scala:216-221 applied to a vector instead of to every entry).  That is half the
//      bytes per step (25 MB instead of 50 MB at N = 2504: resident in both L2 partitions) and no rounding of the N^2
//      centred entries.  v_j goes to row-major VT[i][j]; the block's share of h = V^T y to hpart[b][.];
//   B  h = sum_b hpart[b] (fixed order), y -= V h on the own rows, the share of the second Gram-Schmidt pass to hpart2;
//   C  the same with hpart2, alpha_j = h_j + h2_j, w_out rows = y.
// VT is row-major (n x cap) so that one block's slice is contiguous in the Lanczos index q: the dot products and the
// updates of a block read only its own R rows, coalesced.  Summation orders are fixed: run-to-run deterministic.
constexpr int kLzPersistMaxN = 16384;   // w_in staged in shared memory: 8 n bytes
constexpr int kLzThreads = 1024;
constexpr int kLzSeg = 512;             // columns per warp task of the matvec
constexpr int kLzVtCols = 32;           // leading basis columns of the block's rows that are mirrored in shared memory

struct LzArgs {
    const int32_t* S;
    const double* rowsum;
    const double* scal;     // scal[0] = matrixMean
    double* VT;             // n x cap, row-major
    double* wbuf;           // 2 n
    double* alpha;
    double* beta;
    double* G;              // cap x cap: Gram matrix V^T V of the basis, row j filled at step j (one-reduction Gram-Schmidt)
    double* hpart;          // 2 x blocks x cap
    double* part;           // part[0] = ||w||^2 after the last step (one partial for lz_check_kernel)
    int* st;                // st[0] = next step, st[1] = flag (0 run, 2 breakdown), st[3] = step cap
    unsigned* bar;          // grid barrier counter, zero at launch
    int n, cap, nsteps, pre;
    const int* gate;        // != nullptr: the launch is speculative and returns at once while *gate == 0
    int rows_smem;          // leading rows of every block's share of S that are kept in shared memory for the whole launch
    long long* prof;        // optional (VPCA_LZ_PROF=1): block 0's globaltimer at the phase boundaries of each step, 8 per step
};

// int32 -> double without the (slow) I2F.F64: the bits 0x43300000'(x ^ 0x80000000) are the double 2^52 + 2^31 + x, and one
// exact FP64 subtraction leaves x.
__device__ __forceinline__ double lz_i2d(int x) {
    return __hiloint2double(0x43300000, x ^ (int)0x80000000) - 4503601774854144.0;
}

// Three block-wide sums with one pair of barriers (fixed order: warp shuffles, then the warp totals in warp order).
__device__ __forceinline__ void block_sum3(double& a0, double& a1, double& a2, double* red3) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    a0 = warp_sum(a0);
    a1 = warp_sum(a1);
    a2 = warp_sum(a2);
    __syncthreads();   // protect red3 from the previous use
    if (lane == 0) {
        red3[wid] = a0;
        red3[32 + wid] = a1;
        red3[64 + wid] = a2;
    }
    __syncthreads();
    a0 = warp_sum(lane < nw ? red3[lane] : 0.0);
    a1 = warp_sum(lane < nw ? red3[32 + lane] : 0.0);
    a2 = warp_sum(lane < nw ? red3[64 + lane] : 0.0);
}

__device__ __forceinline__ long long lz_timer() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ void lz_grid_barrier(unsigned* ctr, unsigned& target, unsigned nblocks) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += nblocks;
        __threadfence();
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
        unsigned v;
        const long long t0 = clock64();
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
            if (v < target && clock64() - t0 > 20000000000LL) __trap();   // a block that never arrives must not hang the box
        } while (v < target);
    }
    __syncthreads();
}

// hrow[q] = sum over the block's rows of VT[i0 + r][q] * y[r] for q < jc: this block's share of V^T y.  Few columns
// (the common case: jc <= 128): one warp per column, the rows spread over the lanes -- one L2 latency deep instead of R
// dependent-latency loads per thread; many columns: one thread per column (coalesced across q).  Fixed orders either way.
// Entry (row i0 + r, column q) of the basis: the first kLzVtCols columns of the block's rows are mirrored in shared memory
// (a solve rarely needs more than 16 + 8 + k columns, so the Gram-Schmidt passes run without an L2 round trip).
__device__ __forceinline__ double lz_vt(const LzArgs& a, const double* vts, int i0, int r, int q) {
    return q < kLzVtCols ? vts[r * kLzVtCols + q] : a.VT[(size_t)(i0 + r) * a.cap + q];
}

__device__ __forceinline__ void lz_share(const LzArgs& a, const double* vts, int i0, int R, int jc, const double* y, double* hrow) {
    if (jc <= 128) {
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        for (int q = wid; q < jc; q += kLzThreads / 32) {
            double acc = 0.0;
            for (int r = lane; r < R; r += 32) acc += lz_vt(a, vts, i0, r, q) * y[r];
            acc = warp_sum(acc);
            if (lane == 0) hrow[q] = acc;
        }
    } else {
        for (int q = threadIdx.x; q < jc; q += kLzThreads) {
            double acc = 0.0;
            for (int r = 0; r < R; ++r) acc += lz_vt(a, vts, i0, r, q) * y[r];
            hrow[q] = acc;
        }
    }
}

// dst[q] = sum over the blocks of src[b][q], q < jc.  148 dependent-latency L2 loads per column if one thread walked the
// blocks; instead warp w takes the blocks b = w, w + 32, ... (a handful of independent coalesced loads per lane, 32 columns
// at a time) and the 32 partial sums of a column are added in warp order: deterministic and ~1 L2 latency deep.
// Ends with a block barrier: dst is complete for every thread.
__device__ __forceinline__ void lz_reduce_cols(const LzArgs& a, int nblocks, const double* src, int jc, double* dst, double* red2) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int qc = 0; qc < jc; qc += 32) {
        const int q = qc + lane;
        double acc = 0.0;
        if (q < jc) {
            double p0 = 0.0, p1 = 0.0, p2 = 0.0, p3 = 0.0;
            int b = wid;
            for (; b + 96 < nblocks; b += 128) {
                p0 += __ldcg(src + (size_t)b * a.cap + q);
                p1 += __ldcg(src + (size_t)(b + 32) * a.cap + q);
                p2 += __ldcg(src + (size_t)(b + 64) * a.cap + q);
                p3 += __ldcg(src + (size_t)(b + 96) * a.cap + q);
            }
            for (; b < nblocks; b += 32) p0 += __ldcg(src + (size_t)b * a.cap + q);
            acc = (p0 + p1) + (p2 + p3);
        }
        __syncthreads();                 // red2 of the previous column chunk has been consumed
        red2[wid * 33 + lane] = acc;
        __syncthreads();
        if (wid == 0 && q < jc) {
            double t = 0.0;
#pragma unroll 8
            for (int w2 = 0; w2 < kLzThreads / 32; ++w2) t += red2[w2 * 33 + lane];
            dst[q] = t;
        }
    }
    __syncthreads();
}

// One Gram-Schmidt pass on the rows of this block: hs = sum over blocks of hin (columns [0, jc)), y -= VT hs, and
// (hout != nullptr) this block's share of VT^T y.  Returns hs[jc - 1] (alpha contribution) in every thread.
__device__ __forceinline__ double lz_orth_pass(const LzArgs& a, int nblocks, int i0, int R, int jc, const double* hin,
                                               double* hout, double* hs, double* y, double* red2, const double* vts) {
    lz_reduce_cols(a, nblocks, hin, jc, hs, red2);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int r = wid; r < R; r += kLzThreads / 32) {
        double acc = 0.0;
        for (int q = lane; q < jc; q += 32) acc += lz_vt(a, vts, i0, r, q) * hs[q];
        acc = warp_sum(acc);
        if (lane == 0) y[r] -= acc;
    }
    __syncthreads();
    if (hout != nullptr) lz_share(a, vts, i0, R, jc, y, hout + (size_t)blockIdx.x * a.cap);
    return hs[jc - 1];
}

// Both Gram-Schmidt passes of step j with ONE cross-block reduction.  Classical Gram-Schmidt applied twice computes
// h1 = V^T y, y' = y - V h1, h2 = V^T y', y'' = y' - V h2; but h2 = V^T y - (V^T V) h1 = (I - G) h1 with G = V^T V, and the
// new row of G, g = V^T v_j, can ride on the same reduction as h1 (both are sums of block-local shares).  So every block
// reduces (h1, g), completes its copy of G, forms h = h1 + (I - G) h1 itself and updates y -= V h: one reduction and one
// grid barrier less per step than two explicit passes, the same orthogonality to rounding.  Returns alpha_j = h[j].
__device__ __forceinline__ double lz_fused_pass(const LzArgs& a, int nblocks, int i0, int R, int j, const double* hin,
                                                const double* gin, double* hs, double* gs, double* Gs, double* y,
                                                double* red2, const double* vts) {
    const int jc = j + 1;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (gin == nullptr) {
        // packed shares: columns [0, jc) of hin hold the shares of h1, columns [jc, 2 jc) those of g -- ONE reduction round
        // (for 2 jc <= 32 a single L2 latency) yields both
        lz_reduce_cols(a, nblocks, hin, 2 * jc, hs, red2);
        for (int q = threadIdx.x; q < jc; q += kLzThreads) gs[q] = hs[jc + q];
        __syncthreads();
    } else {
        lz_reduce_cols(a, nblocks, hin, jc, hs, red2);   // h1
        lz_reduce_cols(a, nblocks, gin, jc, gs, red2);   // g = row j of G
    }
    // row / column j of G: every block keeps the leading kLzVtCols x kLzVtCols corner in shared memory, block 0 also
    // writes the full matrix to global memory for the (rare) solves that run past kLzVtCols columns and for later launches
    for (int q = threadIdx.x; q < jc; q += kLzThreads) {
        if (j < kLzVtCols) {
            Gs[j * kLzVtCols + q] = gs[q];
            Gs[q * kLzVtCols + j] = gs[q];
        }
        if (blockIdx.x == 0) {
            a.G[(size_t)j * a.cap + q] = gs[q];
            a.G[(size_t)q * a.cap + j] = gs[q];
        }
    }
    __syncthreads();
    // h = h1 + (I - G) h1 on columns 0 .. j; G(q, j) = g[q] is this step's, older entries come from the mirror / global
    double hq = 0.0;
    const int q0 = threadIdx.x;
    if (q0 < jc) {
        double acc = 0.0;
        for (int p = 0; p < jc; ++p) {
            const double gqp = (p == j) ? gs[q0] : (q0 == j) ? gs[p]
                               : (q0 < kLzVtCols && p < kLzVtCols) ? Gs[q0 * kLzVtCols + p] : __ldcg(a.G + (size_t)q0 * a.cap + p);
            acc += gqp * hs[p];
        }
        hq = hs[q0] + (hs[q0] - acc);
    }
    __syncthreads();
    if (q0 < jc) hs[q0] = hq;
    __syncthreads();
    for (int r = wid; r < R; r += kLzThreads / 32) {
        double acc = 0.0;
        for (int q = lane; q < jc; q += 32) acc += lz_vt(a, vts, i0, r, q) * hs[q];
        acc = warp_sum(acc);
        if (lane == 0) y[r] -= acc;
    }
    __syncthreads();
    return hs[j];
}

__global__ void __launch_bounds__(kLzThreads, 1) lz_persist_kernel(const LzArgs a) {
    extern __shared__ __align__(16) double lzsm[];
    __shared__ double red[33];
    __shared__ double red2[(kLzThreads / 32) * 33];
    __shared__ double red3[96];
    const int n = a.n, nblocks = (int)gridDim.x;
    const int rows_per = (n + nblocks - 1) / nblocks;
    const int i0 = min(n, (int)blockIdx.x * rows_per);
    const int R = min(rows_per, n - i0);
    const int nseg = (n + kLzSeg - 1) / kLzSeg;
    double* wsm = lzsm;                                  // n: w_in
    double* hs = wsm + (((size_t)n + 1) & ~(size_t)1);   // cap
    double* y = hs + a.cap;                              // rows_per
    double* segp = y + ((rows_per + 1) & ~1);            // rows_per x nseg (even offsets keep the int4 rows below 16-byte aligned)
    // The block's rows of S never change: the first rows_smem of them live in shared memory for the whole launch (at
    // N = 2504 all 17 rows, 170 KB), so a step's mat-vec costs no L2 traffic at all for them.
    const int spitch = (n + 3) & ~3;
    double* vts = segp + (((size_t)rows_per * nseg + 1) & ~(size_t)1);   // rows_per x kLzVtCols
    double* rbar_sm = vts + (size_t)rows_per * kLzVtCols;                // n: rowSums / N (VariantsPca.scala:216), once per launch
    double* Gs = rbar_sm + (((size_t)n + 1) & ~(size_t)1);               // kLzVtCols x kLzVtCols corner of G = V^T V
    double* gs = Gs + kLzVtCols * kLzVtCols;                             // cap: the new row of G
    double* vjs = gs + a.cap;                                            // rows_per: the block's rows of v_j
    int32_t* ssm = reinterpret_cast<int32_t*>(vjs + ((rows_per + 1) & ~1));
    const int rs = min(R, a.rows_smem);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const double rc = (double)n;
    const double mm = a.scal[0];
    unsigned target = 0;
    if (a.gate != nullptr && *a.gate == 0) return;
    if (a.st[1] != 0) return;   // every block reads the same flag (nothing in this launch changes it before this point)
    if ((n & 3) == 0) {
        for (int e = threadIdx.x; e < rs * (n >> 2); e += kLzThreads) {
            const int r = e / (n >> 2), c4 = e - r * (n >> 2);
            reinterpret_cast<int4*>(ssm + (size_t)r * spitch)[c4] = __ldg(reinterpret_cast<const int4*>(a.S + (size_t)(i0 + r) * n) + c4);
        }
    } else {
        for (int e = threadIdx.x; e < rs * n; e += kLzThreads) {
            const int r = e / n, c = e - r * n;
            ssm[(size_t)r * spitch + c] = __ldg(a.S + (size_t)(i0 + r) * n + c);
        }
    }
    for (int c = threadIdx.x; c < n; c += kLzThreads) rbar_sm[c] = __ddiv_rn(a.rowsum[c], rc);
    __syncthreads();
    int j = a.st[0];
    for (int e = threadIdx.x; e < R * kLzVtCols; e += kLzThreads) {       // the columns earlier launches (or the lock) wrote
        const int r = e / kLzVtCols, q = e - r * kLzVtCols;
        vts[e] = q < j ? a.VT[(size_t)(i0 + r) * a.cap + q] : 0.0;
    }
    for (int e = threadIdx.x; e < kLzVtCols * kLzVtCols; e += kLzThreads) {   // G of the columns earlier launches built
        const int q = e / kLzVtCols, p2 = e - q * kLzVtCols;
        Gs[e] = (q < j && p2 < j && !a.pre) ? __ldcg(a.G + (size_t)q * a.cap + p2) : 0.0;
    }
    __syncthreads();
    const int jend = min(j + a.nsteps, a.st[3]);
    double* hp1 = a.hpart;
    double* hp2 = a.hpart + (size_t)nblocks * a.cap;

    if (a.pre && j > 0 && j < jend) {
        // deflated restart: G of the j locked columns first (column c against columns 0 .. c: one share + reduction each)
        for (int c = 0; c < j; ++c) {
            for (int r = threadIdx.x; r < R; r += kLzThreads) y[r] = lz_vt(a, vts, i0, r, c);
            __syncthreads();
            lz_share(a, vts, i0, R, c + 1, y, hp2 + (size_t)blockIdx.x * a.cap);
            lz_grid_barrier(a.bar, target, nblocks);
            lz_reduce_cols(a, nblocks, hp2, c + 1, gs, red2);
            for (int q = threadIdx.x; q <= c; q += kLzThreads) {
                if (c < kLzVtCols) {
                    Gs[c * kLzVtCols + q] = gs[q];
                    Gs[q * kLzVtCols + c] = gs[q];
                }
                if (blockIdx.x == 0) {
                    a.G[(size_t)c * a.cap + q] = gs[q];
                    a.G[(size_t)q * a.cap + c] = gs[q];
                }
            }
            lz_grid_barrier(a.bar, target, nblocks);   // hp2 is reused by the next column
        }
        // then the start vector is made orthogonal to the j locked columns (two explicit passes) before step j
        double* w_in = a.wbuf + (size_t)(j & 1) * n;
        for (int r = threadIdx.x; r < R; r += kLzThreads) y[r] = w_in[i0 + r];
        __syncthreads();
        for (int pass = 0; pass < 2; ++pass) {
            double* hp = pass == 0 ? hp1 : hp2;
            lz_share(a, vts, i0, R, j, y, hp + (size_t)blockIdx.x * a.cap);
            lz_grid_barrier(a.bar, target, nblocks);
            lz_orth_pass(a, nblocks, i0, R, j, hp, nullptr, hs, y, red2, vts);
        }
        for (int r = threadIdx.x; r < R; r += kLzThreads) w_in[i0 + r] = y[r];
        lz_grid_barrier(a.bar, target, nblocks);
    }

    bool broke = false;
    for (; j < jend; ++j) {
        const double* w_in = a.wbuf + (size_t)(j & 1) * n;
        double* w_out = a.wbuf + (size_t)((j + 1) & 1) * n;
        // ---- phase A: stage w_in, beta_j, y = C v_j on the own rows, share of V^T y
        const bool prof = a.prof != nullptr && blockIdx.x == 0 && threadIdx.x == 0 && j < 32;
        if (prof) a.prof[j * 8 + 0] = lz_timer();
        double s0 = 0.0, s1 = 0.0, s2 = 0.0;
        for (int c0 = threadIdx.x; c0 < n; c0 += 4 * kLzThreads) {
            double wv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {   // the (up to) four L2 loads of a thread are in flight together
                const int c = c0 + u * kLzThreads;
                wv[u] = c < n ? __ldcg(w_in + c) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int c = c0 + u * kLzThreads;
                if (c < n) {
                    wsm[c] = wv[u];
                    s0 += wv[u] * wv[u];
                    s1 += wv[u];
                    s2 += rbar_sm[c] * wv[u];
                }
            }
        }
        block_sum3(s0, s1, s2, red3);   // (syncs: wsm is complete)
        if (prof) a.prof[j * 8 + 1] = lz_timer();
        const double nrm = sqrt(s0);
        if (!(nrm > 0.0) || !(nrm <= DBL_MAX)) {   // exact breakdown or non-finite: every block sees the same value
            broke = true;
            break;
        }
        const double inv = 1.0 / nrm;
        const bool vec4 = (n & 3) == 0;
        // column workers x row groups must fill most of the 32 warps (5 x 6 at N = 2504, 8 x 4 at 4096); cohorts whose segment
        // count leaves more than a fifth of them idle (e.g. 20 segments at N = 10 000) use the (row, segment) task list below
        const int CWp = min(nseg, kLzThreads / 32), Gp = (kLzThreads / 32) / CWp;
        const bool regw = vec4 && 5 * CWp * Gp >= 4 * (kLzThreads / 32);
        if (regw) {
            // A warp keeps ONE 512-column segment of w in registers (16 doubles per lane) and walks rows of S under it:
            // per element only the 4 bytes of S are read again (shared memory or L2), not the 8 bytes of w as well.
            // Column workers cw = 0 .. CW-1 own the segments cw, cw + CW, ...; G = 32 / CW row groups share the rows.
            const int CW = min(nseg, kLzThreads / 32), G = (kLzThreads / 32) / CW;
            const int cw = wid % CW, g = wid / CW;
            if (g < G) {
                for (int sg = cw; sg < nseg; sg += CW) {
                    const int c0 = sg * kLzSeg, c1 = min(n, c0 + kLzSeg);
                    double2 wa[kLzSeg / 128], wb[kLzSeg / 128];
#pragma unroll
                    for (int u = 0; u < kLzSeg / 128; ++u) {
                        const int c = c0 + (u * 32 + lane) * 4;
                        if (c < c1) {
                            wa[u] = *reinterpret_cast<const double2*>(wsm + c);
                            wb[u] = *reinterpret_cast<const double2*>(wsm + c + 2);
                        } else {
                            wa[u] = make_double2(0.0, 0.0);
                            wb[u] = make_double2(0.0, 0.0);
                        }
                    }
                    for (int r = g; r < R; r += G) {
                        const bool in_smem = r < rs;
                        const int32_t* srow = in_smem ? ssm + (size_t)r * spitch : a.S + (size_t)(i0 + r) * n;
                        double p[kLzSeg / 128];
#pragma unroll
                        for (int u = 0; u < kLzSeg / 128; ++u) {
                            const int c = c0 + (u * 32 + lane) * 4;
                            p[u] = 0.0;
                            if (c < c1) {
                                const int4 sv = in_smem ? *reinterpret_cast<const int4*>(srow + c)
                                                        : __ldg(reinterpret_cast<const int4*>(srow + c));
                                p[u] = lz_i2d(sv.x) * wa[u].x + lz_i2d(sv.y) * wa[u].y + (lz_i2d(sv.z) * wb[u].x + lz_i2d(sv.w) * wb[u].y);
                            }
                        }
                        double acc = (p[0] + p[1]) + (p[2] + p[3]);
                        acc = warp_sum(acc);
                        if (lane == 0) segp[r * nseg + sg] = acc;
                    }
                }
            }
        } else if (vec4) {
            for (int task = wid; task < R * nseg; task += kLzThreads / 32) {
                const int r = task / nseg, sg = task - r * nseg;
                const bool in_smem = r < rs;
                const int32_t* srow = in_smem ? ssm + (size_t)r * spitch : a.S + (size_t)(i0 + r) * n;
                const int c0 = sg * kLzSeg, c1 = min(n, c0 + kLzSeg);
                double p[kLzSeg / 128];
#pragma unroll
                for (int u = 0; u < kLzSeg / 128; ++u) {
                    const int c = c0 + (u * 32 + lane) * 4;
                    p[u] = 0.0;
                    if (c < c1) {
                        const int4 sv = in_smem ? *reinterpret_cast<const int4*>(srow + c)
                                                : __ldg(reinterpret_cast<const int4*>(srow + c));
                        const double2 wa = *reinterpret_cast<const double2*>(wsm + c);
                        const double2 wb = *reinterpret_cast<const double2*>(wsm + c + 2);
                        p[u] = lz_i2d(sv.x) * wa.x + lz_i2d(sv.y) * wa.y + (lz_i2d(sv.z) * wb.x + lz_i2d(sv.w) * wb.y);
                    }
                }
                double acc = (p[0] + p[1]) + (p[2] + p[3]);
                acc = warp_sum(acc);
                if (lane == 0) segp[r * nseg + sg] = acc;
            }
        } else {
            for (int task = wid; task < R * nseg; task += kLzThreads / 32) {
                const int r = task / nseg, sg = task - r * nseg;
                const bool in_smem = r < rs;
                const int32_t* srow = in_smem ? ssm + (size_t)r * spitch : a.S + (size_t)(i0 + r) * n;
                const int c0 = sg * kLzSeg, c1 = min(n, c0 + kLzSeg);
                double acc = 0.0;
                for (int c = c0 + lane; c < c1; c += 32) acc += (double)(in_smem ? srow[c] : __ldg(srow + c)) * wsm[c];
                acc = warp_sum(acc);
                if (lane == 0) segp[r * nseg + sg] = acc;
            }
        }
        __syncthreads();
        if (prof) a.prof[j * 8 + 2] = lz_timer();
        for (int r = threadIdx.x; r < R; r += kLzThreads) {
            double acc = 0.0;
            for (int sg = 0; sg < nseg; ++sg) acc += segp[r * nseg + sg];
            y[r] = (acc - rbar_sm[i0 + r] * s1 - s2 + mm * s1) * inv;
            const double vj = wsm[i0 + r] * inv;
            a.VT[(size_t)(i0 + r) * a.cap + j] = vj;
            if (j < kLzVtCols) vts[r * kLzVtCols + j] = vj;
            vjs[r] = vj;
        }
        __syncthreads();
        if (prof) a.prof[j * 8 + 3] = lz_timer();
        const bool packed = 2 * (j + 1) <= a.cap;   // both shares side by side in one buffer: one reduction round later
        lz_share(a, vts, i0, R, j + 1, y, hp1 + (size_t)blockIdx.x * a.cap);     // share of h1 = V^T y
        lz_share(a, vts, i0, R, j + 1, vjs, (packed ? hp1 + (j + 1) : hp2) + (size_t)blockIdx.x * a.cap);   // share of g = V^T v_j
        if (prof) a.prof[j * 8 + 4] = lz_timer();
        lz_grid_barrier(a.bar, target, nblocks);
        // ---- phase B: both Gram-Schmidt passes from one reduction (lz_fused_pass)
        if (prof) a.prof[j * 8 + 5] = lz_timer();
        const double aj = lz_fused_pass(a, nblocks, i0, R, j, hp1, packed ? nullptr : hp2, hs, gs, Gs, y, red2, vts);
        if (prof) a.prof[j * 8 + 6] = lz_timer();
        for (int r = threadIdx.x; r < R; r += kLzThreads) w_out[i0 + r] = y[r];
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            a.alpha[j] = aj;
            a.beta[j] = nrm;
        }
        if (prof) a.prof[j * 8 + 7] = lz_timer();
        lz_grid_barrier(a.bar, target, nblocks);
    }
    if (blockIdx.x == 0) {
        // ||w||^2 of the vector the next step would normalise: what lz_check_kernel turns into the residual bound
        const double* w_last = a.wbuf + (size_t)(j & 1) * n;
        double s0 = 0.0;
        if (!broke)
            for (int c = threadIdx.x; c < n; c += kLzThreads) {
                const double wv = __ldcg(w_last + c);
                s0 += wv * wv;
            }
        s0 = block_sum(s0, red);
        if (threadIdx.x == 0) {
            a.part[0] = s0;
            a.st[0] = j;
            if (broke) a.st[1] = 2;
        }
    }
}

// One thread, right after lz_check_kernel: converged (st[1] == 1) arms the deflated re-run that is already enqueued behind it
// (st[4] = 1, step window [k, k + vsteps), flag back to "running"); otherwise st[4] = 0 and every kernel of that re-run
// returns at once, leaving the state of the main run untouched for the next chunk.
__global__ void lz_gate_kernel(int* __restrict__ st, int k, int vsteps) {
    if (st[1] == 1) {
        st[4] = 1;
        st[0] = k;
        st[1] = 0;
        st[3] = k + vsteps;
    } else {
        st[4] = 0;
    }
}

// Z[:, c] = VT Y[:, c] for the row-major basis: one warp per (row, c).
__global__ void __launch_bounds__(256) lz_ritz_rm_kernel(const double* __restrict__ VT, int n, int cap,
                                                         const double* __restrict__ Y, int m, int k, double* __restrict__ Z,
                                                         const int* __restrict__ gate = nullptr) {
    if (gate != nullptr && *gate == 0) return;
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= n) return;
    const double* __restrict__ vt = VT + (size_t)row * cap;
    for (int c = 0; c < k; ++c) {
        const double* __restrict__ yc = Y + (size_t)c * m;
        double acc = 0.0;
        for (int q = lane; q < m; q += 32) acc += vt[q] * yc[q];
        acc = warp_sum(acc);
        if (lane == 0) Z[(size_t)c * n + row] = acc;
    }
}

// VT[:, 0..k) = Z (the converged Ritz vectors become the locked leading columns of the deflated run)
__global__ void lz_lock_kernel(double* __restrict__ VT, int n, int cap, const double* __restrict__ Z, int k,
                               const int* __restrict__ gate = nullptr) {
    if (gate != nullptr && *gate == 0) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int c = 0; c < k; ++c) VT[(size_t)i * cap + c] = Z[(size_t)c * n + i];
}

// ------------------------------------------------------------------------------------------ projection
// Coordinates of projected samples on the fitted PCs (Gower's add-a-point formula, the Nystrom extension of the centred
// similarity): the cross row X_p (counts shared with every fitted sample, int32) is centred with the FITTED statistics in
// the operation order of center_kernel (VariantsPca.scala:216-221 applied to a new row),
//   c_pf = ((X_pf - rowMean_p) - rowSums_f / N) + matrixMean,   rowMean_p = (sum_f X_pf) / N,
// and y_pc = (sum_f c_pf u_fc) / lambda_c.  Three launches, every reduction in a fixed order (no atomics): two calls give
// bit-identical output.  The cross block is read twice -- the row sums must precede the centring -- but the second read
// comes from L2 (the block of 2504 x 2504 counts is 25 MB).
constexpr int kProjCols = 128;   // columns of S per block: 4 per lane, so a cohort of N samples makes ceil(N / 128) column
                                 // chunks and even 50 projected rows fill ~140 blocks at N = 2504
constexpr int kProjRows = 8;     // cross rows per block, one warp each

__global__ void proj_rowmean_kernel(const int32_t* __restrict__ X, int n, int m, double* __restrict__ rowmean) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= m) return;
    const int32_t* r = X + (size_t)row * n;
    long long acc = 0;
    for (int j = lane; j < n; j += 32) acc += r[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    // exact integer sum (the foldLeft(0D) of :206 on the new row), then rowMean as center_kernel forms it
    if (lane == 0) rowmean[row] = __ddiv_rn((double)acc, (double)n);
}

// part[(q * m + p) * k + c] = sum over the columns f of chunk q of c_pf u_fc (ascending f per lane, then a fixed xor tree)
__global__ void __launch_bounds__(32 * kProjRows) proj_dot_kernel(const int32_t* __restrict__ X, int n, int m,
                                                                  const double* __restrict__ rowsum,
                                                                  const double* __restrict__ mm,
                                                                  const double* __restrict__ rowmean,
                                                                  const double* __restrict__ U, int k,
                                                                  double* __restrict__ part) {
    const int q = blockIdx.x;
    const int p = blockIdx.y * kProjRows + (int)(threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (p >= m) return;
    const double rc = (double)n, rm = rowmean[p], mean = mm[0];
    constexpr int kPer = kProjCols / 32;
    double cv[kPer];
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
        const int f = q * kProjCols + i * 32 + lane;
        cv[i] = 0.0;
        if (f < n) {
            const double data = lz_i2d(X[(size_t)p * n + f]);
            cv[i] = __dadd_rn(__dsub_rn(__dsub_rn(data, rm), __ddiv_rn(rowsum[f], rc)), mean);
        }
    }
    for (int c = 0; c < k; ++c) {
        const double* u = U + (size_t)c * n;
        double acc = 0.0;
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
            const int f = q * kProjCols + i * 32 + lane;
            if (f < n) acc = __fma_rn(cv[i], u[f], acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) part[((size_t)q * m + p) * k + c] = acc;
    }
}

// y[p + c * m] = (sum over chunks q in ascending order of part) / lambda_c
__global__ void proj_finish_kernel(const double* __restrict__ part, int chunks, int m, int k,
                                   const double* __restrict__ evals, double* __restrict__ y) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m * k) return;
    const int p = t / k, c = t - p * k;
    double acc = 0.0;
    for (int q = 0; q < chunks; ++q) acc = __dadd_rn(acc, part[((size_t)q * m + p) * k + c]);
    y[p + (size_t)c * m] = __ddiv_rn(acc, evals[c]);
}

}  // namespace

int proj_chunks(int n) { return (n + kProjCols - 1) / kProjCols; }

cudaError_t eig_project(const EigWork& w, const int32_t* d_X, int m, int k, double* d_rowmean, double* d_part, double* d_y,
                        cudaStream_t stream) {
    if (m <= 0) return cudaSuccess;
    const int n = w.n, chunks = proj_chunks(n);
    proj_rowmean_kernel<<<(m + 7) / 8, 256, 0, stream>>>(d_X, n, m, d_rowmean);
    proj_dot_kernel<<<dim3(chunks, (m + kProjRows - 1) / kProjRows), 32 * kProjRows, 0, stream>>>(
        d_X, n, m, w.d_rowsum, w.d_mm, d_rowmean, w.d_evecs, k, d_part);
    proj_finish_kernel<<<(m * k + 255) / 256, 256, 0, stream>>>(d_part, chunks, m, k, w.d_evals, d_y);
    return cudaGetLastError();
}

cudaError_t eig_alloc(EigWork& w, int n, int kmax) {
    w.n = n;
    w.kmax = kmax;
    cudaError_t e;
#define VPCA_TRY(x) if ((e = (x)) != cudaSuccess) return e
    VPCA_TRY(cudaMalloc(&w.d_C, (size_t)n * n * sizeof(double)));
    VPCA_TRY(cudaMalloc(&w.d_rowsum, (size_t)n * sizeof(double)));
    VPCA_TRY(cudaMalloc(&w.d_v, 2 * (size_t)n * sizeof(double)));   // vprev / vcur ping-pong
    VPCA_TRY(cudaMalloc(&w.d_w, (size_t)n * sizeof(double)));
    VPCA_TRY(cudaMalloc(&w.d_p, 2 * (size_t)n * sizeof(double)));   // p ping-pong (fused step kernel)
    VPCA_TRY(cudaMalloc(&w.d_diag, (size_t)n * sizeof(double)));
    VPCA_TRY(cudaMalloc(&w.d_off, 2 * (size_t)n * sizeof(double)));   // e and e^2
    VPCA_TRY(cudaMalloc(&w.d_tau, (size_t)n * sizeof(double)));
    VPCA_TRY(cudaMalloc(&w.d_scal, 16 * sizeof(double)));
    VPCA_TRY(cudaMalloc(&w.d_mm, sizeof(double)));
    VPCA_TRY(cudaMalloc(&w.d_evals, (size_t)kmax * sizeof(double)));
    VPCA_TRY(cudaMalloc(&w.d_evecs, (size_t)n * kmax * sizeof(double)));
    VPCA_TRY(cudaMalloc(&w.d_lu, 8 * (size_t)n * sizeof(double)));
    VPCA_TRY(cudaMalloc(&w.d_nz, sizeof(int)));
    VPCA_TRY(cudaMalloc(&w.d_step, 4 * sizeof(int)));   // {next, current step, ticket counter, -}
#undef VPCA_TRY
    return cudaSuccess;
}

void eig_free(EigWork& w) {
    cudaFree(w.d_C); cudaFree(w.d_rowsum); cudaFree(w.d_v); cudaFree(w.d_w); cudaFree(w.d_p);
    cudaFree(w.d_diag); cudaFree(w.d_off); cudaFree(w.d_tau); cudaFree(w.d_scal); cudaFree(w.d_mm); cudaFree(w.d_evals);
    cudaFree(w.d_evecs); cudaFree(w.d_lu); cudaFree(w.d_nz); cudaFree(w.d_step);
    cudaFree(w.d_V); cudaFree(w.d_lzw); cudaFree(w.d_lzs); cudaFree(w.d_lzst); cudaFree(w.d_lzbar); cudaFree(w.d_lzprof); cudaFree(w.d_lzG);
    if (w.graph_exec != nullptr) cudaGraphExecDestroy(w.graph_exec);
    if (w.lz_graph != nullptr) cudaGraphExecDestroy(w.lz_graph);
    w = EigWork{};
}

cudaError_t center_gram(EigWork& w, const int32_t* d_S, cudaStream_t stream, bool materialise) {
    const int n = w.n;
    w.d_S = d_S;   // the persistent Lanczos applies the centring to vectors and reads the int32 Gram itself
    rowsum_kernel<<<(n + 7) / 8, 256, 0, stream>>>(d_S, n, w.d_rowsum);
    matrix_mean_kernel<<<1, 1024, 0, stream>>>(w.d_rowsum, n, w.d_scal, w.d_nz, w.d_mm);
    w.c_valid = false;
    if (materialise) return center_matrix(w, stream);
    return cudaGetLastError();
}

// C = S - rowMean - colMean + matrixMean as an FP64 matrix (VariantsPca.scala:216-221): what vpca_get_centered returns and
// what the direct reduction and the five-kernel Lanczos read.  The persistent Lanczos never needs it (50 MB at N = 2504).
cudaError_t center_matrix(EigWork& w, cudaStream_t stream) {
    if (w.c_valid) return cudaSuccess;
    const int n = w.n;
    const int bx = (n + 1023) / 1024 < 1 ? 1 : (n + 1023) / 1024;
    center_kernel<<<dim3(bx, n), 256, 0, stream>>>(w.d_S, w.d_rowsum, w.d_scal, n, w.d_C);
    w.c_valid = true;
    return cudaGetLastError();
}

// Top-k by Lanczos.  *used = true: d_evals / d_evecs hold the answer.  *used = false: the caller runs the direct
// solver (C is untouched).  Synchronises the stream once per kLzChunk steps to read the residual.
static cudaError_t lanczos_topk(EigWork& w, int k, cudaStream_t stream, int64_t* launches, bool* used) {
    *used = false;
    const int n = w.n;
    const int npart = (n + 31) / 32;
    const int kmax = w.kmax;
    cudaError_t e;
#define VPCA_TRY(x) if ((e = (x)) != cudaSuccess) return e
    if (w.d_V == nullptr) {
        // persistent form: one 1024-thread block per SM, launched cooperatively (all blocks co-resident)
        int dev = 0, sms = 0, coop = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
        const char* lp = getenv("VPCA_LZ_PERSIST");
        w.lz_blocks = (coop != 0 && sms > 0 && !(lp != nullptr && atoi(lp) == 0)) ? sms : 0;
    }
    const size_t small_doubles = 5 * (size_t)kLzCap + (size_t)kLzCap * kmax + 16 + 4 + 16 + (size_t)npart +
                                 2 * (size_t)w.lz_blocks * kLzCap;
    if (w.d_V == nullptr) {
        VPCA_TRY(cudaMalloc(&w.d_V, (size_t)n * kLzCap * sizeof(double)));
        VPCA_TRY(cudaMalloc(&w.d_lzw, 2 * (size_t)n * sizeof(double)));
        VPCA_TRY(cudaMalloc(&w.d_lzs, small_doubles * sizeof(double)));
        VPCA_TRY(cudaMalloc(&w.d_lzst, 8 * sizeof(int)));
        VPCA_TRY(cudaMemset(w.d_lzst, 0, 8 * sizeof(int)));
        VPCA_TRY(cudaMalloc(&w.d_lzbar, sizeof(unsigned)));
        VPCA_TRY(cudaMalloc(&w.d_lzG, (size_t)kLzCap * kLzCap * sizeof(double)));
        VPCA_TRY(cudaMemset(w.d_lzG, 0, (size_t)kLzCap * kLzCap * sizeof(double)));
        if (const char* pf = getenv("VPCA_LZ_PROF"); pf != nullptr && atoi(pf) != 0) {
            VPCA_TRY(cudaMalloc(&w.d_lzprof, 64 * 4 * sizeof(long long)));
            VPCA_TRY(cudaMemset(w.d_lzprof, 0, 64 * 4 * sizeof(long long)));
        }
    }
    double* alpha = w.d_lzs;
    double* beta = alpha + kLzCap;
    double* h1 = beta + kLzCap;
    double* h2 = h1 + kLzCap;
    double* e2 = h2 + kLzCap;
    double* Y = e2 + kLzCap;
    double* theta2 = Y + (size_t)kLzCap * kmax;
    double* res = theta2 + 16;
    double* scal2 = res + 4;
    double* part = scal2 + 16;
    int64_t nl = 0;
    const int upd_blocks = npart, mv_blocks = (n + 3) / 4;
    // persistent form: one cooperative launch per chunk (see lz_persist_kernel); the five-kernel graph is kept for
    // cohorts whose start vector does not fit shared memory and as VPCA_LZ_PERSIST=0
    const bool persist = w.lz_blocks > 0 && n <= kLzPersistMaxN;
    double* hpart = part + npart;
    const int rows_per = persist ? (n + w.lz_blocks - 1) / w.lz_blocks : 0;
    const size_t base_smem =
        ((((size_t)n + 1) & ~(size_t)1) + kLzCap + (((size_t)rows_per + 1) & ~(size_t)1) +
         ((((size_t)rows_per * ((n + kLzSeg - 1) / kLzSeg)) + 1) & ~(size_t)1) + (size_t)rows_per * kLzVtCols + (((size_t)n + 1) & ~(size_t)1) +
         (size_t)kLzVtCols * kLzVtCols + kLzCap + (((size_t)rows_per + 1) & ~(size_t)1)) * sizeof(double);
    // what is left of the 227 KB a block may use (minus the kernel's ~9 KB of static shared memory) holds rows of S
    int rows_smem = 0;
    {
        const size_t budget = 232448 - 10240 - 1024;
        const size_t row_bytes = (size_t)((n + 3) & ~3) * sizeof(int32_t);
        if (persist && base_smem < budget) rows_smem = (int)std::min<size_t>((size_t)rows_per, (budget - base_smem) / row_bytes);
        if (const char* sr = getenv("VPCA_LZ_SROWS"); sr != nullptr) rows_smem = std::min(rows_smem, std::max(0, atoi(sr)));
    }
    const size_t persist_smem = base_smem + (size_t)rows_smem * ((n + 3) & ~3) * sizeof(int32_t);
    if (persist) VPCA_TRY(cudaFuncSetAttribute(lz_persist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)persist_smem));
    auto run_chunk = [&](int pre, const int* gate = nullptr) -> cudaError_t {
        if (!persist) {
            nl += 5 * kLzChunk;
            return cudaGraphLaunch(w.lz_graph, stream);
        }
        cudaError_t ce = cudaMemsetAsync(w.d_lzbar, 0, sizeof(unsigned), stream);
        if (ce != cudaSuccess) return ce;
        LzArgs a{};
        a.S = w.d_S;
        a.rowsum = w.d_rowsum;
        a.scal = w.d_scal;
        a.VT = w.d_V;
        a.wbuf = w.d_lzw;
        a.alpha = alpha;
        a.beta = beta;
        a.hpart = hpart;
        a.G = w.d_lzG;
        a.part = part;
        a.st = w.d_lzst;
        a.bar = w.d_lzbar;
        a.n = n;
        a.cap = kLzCap;
        a.nsteps = kLzChunk;
        a.pre = pre;
        a.gate = gate;
        a.rows_smem = rows_smem;
        a.prof = w.d_lzprof;
        void* params[] = {&a};
        nl += 1;
        return cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(lz_persist_kernel), dim3((unsigned)w.lz_blocks),
                                           dim3(kLzThreads), params, persist_smem, stream);
    };

    if (!persist) VPCA_TRY(center_matrix(w, stream));   // the five-kernel form reads the FP64 matrix
    if (!persist && w.lz_graph == nullptr) {
        cudaGraph_t graph = nullptr;
        VPCA_TRY(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
        for (int g = 0; g < kLzChunk; ++g) {
            lz_matvec_kernel<<<mv_blocks, 256, 0, stream>>>(w.d_C, n, w.d_V, w.d_lzw, part, npart, beta, w.d_lzst);
            lz_dots_kernel<<<kLzCap, 128, 0, stream>>>(w.d_V, n, w.d_lzw, h1, w.d_lzst);
            lz_update_kernel<<<upd_blocks, 256, 0, stream>>>(w.d_V, n, w.d_lzw, h1, alpha, part, w.d_lzst, 1);
            lz_dots_kernel<<<kLzCap, 128, 0, stream>>>(w.d_V, n, w.d_lzw, h2, w.d_lzst);
            lz_update_kernel<<<upd_blocks, 256, 0, stream>>>(w.d_V, n, w.d_lzw, h2, alpha, part, w.d_lzst, 2);
        }
        VPCA_TRY(cudaStreamEndCapture(stream, &graph));
        e = cudaGraphInstantiate(&w.lz_graph, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) return e;
    }
    VPCA_TRY(cudaFuncSetAttribute(invit_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));

    const double tol = 1e-12;
    int max_iter = kLzMaxIter;
    if (const char* mi = getenv("VPCA_EIG_MAXIT")) max_iter = std::max(kLzChunk, std::min(kLzMaxIter, atoi(mi)));
    int hst[8] = {0, 0, 0, max_iter, 0, 0, 0, 0};
    double hres[2] = {0.0, 0.0};
    const int vsteps = persist ? kLzVerify : kLzChunk;
    const char* spe = getenv("VPCA_LZ_SPECULATE");
    const bool speculate = persist && k + kLzChunk < n && !(spe != nullptr && atoi(spe) == 0);
    VPCA_TRY(cudaMemcpyAsync(w.d_lzst, hst, sizeof(hst), cudaMemcpyHostToDevice, stream));
    lz_init_kernel<<<npart, 32, 0, stream>>>(w.d_lzw, n, 0x5eedULL, part);
    nl += 1;
    int m = 0, m_prev = 0;
    bool converged = false;
    double rho_prev = 0.0;
    const int max_chunks = std::min(max_iter, n - 1) / kLzChunk;
    for (int chunk = 1; chunk <= max_chunks; ++chunk) {
        VPCA_TRY(run_chunk(0));
        m = chunk * kLzChunk;
        // look at the residual after every replay up to 64 steps, then after every other one
        if (chunk > 4 && (chunk & 1) && chunk != max_chunks) continue;
        bisect_kernel<<<k, 256, 0, stream>>>(alpha, beta + 1, m, e2, w.d_evals, w.d_scal);
        // a tridiagonal matrix of a few dozen rows: one warp (its block-wide reductions then cost no barrier latency)
        invit_kernel<true><<<1, m <= 128 ? 32 : 256, 8 * (size_t)m * sizeof(double), stream>>>(alpha, beta + 1, m, k, w.d_evals, w.d_scal,
                                                                                w.d_lu, Y);
        lz_check_kernel<<<1, 32, 0, stream>>>(part, persist ? 1 : npart, Y, m, k, w.d_scal, w.d_lzst, res, tol);
        nl += 3;
        const bool spec = speculate && chunk == 1;
        if (spec) {
            // The usual case converges at the first test.  Everything that follows a successful test -- Ritz vectors,
            // locking them, the deflated re-run and its verdict -- is enqueued NOW behind a one-thread gate, so the host
            // synchronises once per solve; had the test failed, every gated kernel returns at once and the main run
            // goes on below with its state untouched.
            const int* gate = w.d_lzst + 4;
            lz_gate_kernel<<<1, 1, 0, stream>>>(w.d_lzst, k, vsteps);
            lz_ritz_rm_kernel<<<(n + 7) / 8, 256, 0, stream>>>(w.d_V, n, kLzCap, Y, m, k, w.d_evecs, gate);
            lz_finish_kernel<<<k, 512, 0, stream>>>(w.d_evecs, n, gate);
            lz_lock_kernel<<<(n + 255) / 256, 256, 0, stream>>>(w.d_V, n, kLzCap, w.d_evecs, k, gate);
            lz_init_kernel<<<npart, 32, 0, stream>>>(w.d_lzw + (size_t)(k & 1) * n, n, 0xfaceULL, part, gate);
            VPCA_TRY(run_chunk(1, gate));
            bisect_kernel<<<1, 256, 0, stream>>>(alpha + k, beta + k + 1, vsteps, e2, theta2, scal2, gate);
            lz_verify_kernel<<<1, 1, 0, stream>>>(w.d_evals, k, theta2, w.d_scal, w.d_lzst, gate);
            nl += 7;
        }
        VPCA_TRY(cudaMemcpyAsync(hst, w.d_lzst, sizeof(hst), cudaMemcpyDeviceToHost, stream));
        VPCA_TRY(cudaMemcpyAsync(hres, res, sizeof(hres), cudaMemcpyDeviceToHost, stream));
        VPCA_TRY(cudaStreamSynchronize(stream));
        if (spec && hst[4] == 1) {   // converged at the first test; the re-run has delivered its verdict in st[1]
            w.last_iters = m;
            if (launches) *launches += nl;
            if (hst[1] != 1) return cudaGetLastError();   // missed eigenvalue (3) or breakdown (2): the caller falls back
            *used = true;
            return cudaGetLastError();
        }
        if (hst[1] == 1) {
            converged = true;
            break;
        }
        if (hst[1] != 0) break;   // breakdown
        const double rho = hres[0];
        if (m >= 96 && rho > 1e-3) break;   // no separated top of the spectrum: hopeless within kLzMaxIter
        if (m_prev >= 32 && rho < rho_prev) {
            const double rate = std::log(rho_prev / rho) / (m - m_prev);
            if (m + 1.5 * std::log(rho / tol) / rate > max_iter + 2 * kLzChunk) break;
        }
        rho_prev = rho;
        m_prev = m;
    }
    w.last_iters = m;
    if (launches) *launches += nl;
    if (!converged) return cudaGetLastError();
    nl = 0;

    // Ritz vectors, unit norm, sign rule
    if (persist) lz_ritz_rm_kernel<<<(n + 7) / 8, 256, 0, stream>>>(w.d_V, n, kLzCap, Y, m, k, w.d_evecs);
    else lz_ritz_kernel<<<dim3(npart, k), 256, 0, stream>>>(w.d_V, n, Y, m, w.d_evecs);
    lz_finish_kernel<<<k, 512, 0, stream>>>(w.d_evecs, n);
    nl += 2;

    // Guard against a missed copy of a multiple eigenvalue (a single Krylov sequence sees one vector per eigenspace):
    // lock the k Ritz vectors as the first k basis columns and run one more chunk from a fresh start vector that is
    // orthogonal to them.  Its top Ritz value is a lower bound of the largest eigenvalue of the deflated operator.
    if (k + kLzChunk < n) {
        if (persist) {
            lz_lock_kernel<<<(n + 255) / 256, 256, 0, stream>>>(w.d_V, n, kLzCap, w.d_evecs, k);
            int vst[4] = {k, 0, 0, k + vsteps};
            VPCA_TRY(cudaMemcpyAsync(w.d_lzst, vst, sizeof(vst), cudaMemcpyHostToDevice, stream));
            lz_init_kernel<<<npart, 32, 0, stream>>>(w.d_lzw + (size_t)(k & 1) * n, n, 0xfaceULL, part);
            nl += 2;
            VPCA_TRY(run_chunk(1));   // orthogonalises the start vector against the locked columns, then kLzChunk steps
        } else {
            VPCA_TRY(cudaMemcpyAsync(w.d_V, w.d_evecs, (size_t)n * k * sizeof(double), cudaMemcpyDeviceToDevice, stream));
            int vst[4] = {k - 1, 0, 0, k + kLzChunk};
            VPCA_TRY(cudaMemcpyAsync(w.d_lzst, vst, sizeof(vst), cudaMemcpyHostToDevice, stream));
            lz_init_kernel<<<npart, 32, 0, stream>>>(w.d_lzw + (size_t)(k & 1) * n, n, 0xfaceULL, part);
            lz_dots_kernel<<<kLzCap, 128, 0, stream>>>(w.d_V, n, w.d_lzw, h1, w.d_lzst);
            lz_update_kernel<<<upd_blocks, 256, 0, stream>>>(w.d_V, n, w.d_lzw, h1, alpha, part, w.d_lzst, 1);
            lz_dots_kernel<<<kLzCap, 128, 0, stream>>>(w.d_V, n, w.d_lzw, h2, w.d_lzst);
            lz_update_kernel<<<upd_blocks, 256, 0, stream>>>(w.d_V, n, w.d_lzw, h2, alpha, part, w.d_lzst, 2);
            nl += 5;
            VPCA_TRY(run_chunk(0));
        }
        bisect_kernel<<<1, 256, 0, stream>>>(alpha + k, beta + k + 1, vsteps, e2, theta2, scal2);
        lz_verify_kernel<<<1, 1, 0, stream>>>(w.d_evals, k, theta2, w.d_scal, w.d_lzst);
        nl += 2;
        VPCA_TRY(cudaMemcpyAsync(hst, w.d_lzst, sizeof(hst), cudaMemcpyDeviceToHost, stream));
        VPCA_TRY(cudaStreamSynchronize(stream));
        if (launches) *launches += nl;
        if (hst[1] != 1) return cudaGetLastError();
    } else if (launches) {
        *launches += nl;
    }
#undef VPCA_TRY
    *used = true;
    return cudaGetLastError();
}

cudaError_t eig_topk(EigWork& w, int k, cudaStream_t stream, int64_t* launches) {
    const int n = w.n;
    if (k < 1 || k > w.kmax || k > n) return cudaErrorInvalidValue;
    w.last_method = 1;
    w.last_iters = 0;
    if (w.mode != 1 && n >= (w.mode == 2 ? kLzForcedMinN : kLzMinN)) {
        bool used = false;
        cudaError_t le = lanczos_topk(w, k, stream, launches, &used);
        if (le != cudaSuccess) return le;
        if (used) {
            w.last_method = 2;
            return cudaSuccess;
        }
        w.last_method = 3;
    }
    cudaError_t e = center_matrix(w, stream);   // the reduction works on (and overwrites) the FP64 matrix
    if (e != cudaSuccess) return e;
    w.c_valid = false;
    e = cudaMemsetAsync(w.d_v, 0, 2 * (size_t)n * sizeof(double), stream);
    if (e != cudaSuccess) return e;
    cudaMemsetAsync(w.d_w, 0, (size_t)n * sizeof(double), stream);
    cudaMemsetAsync(w.d_p, 0, 2 * (size_t)n * sizeof(double), stream);
    cudaMemsetAsync(w.d_tau, 0, (size_t)n * sizeof(double), stream);
    cudaMemsetAsync(w.d_off, 0, 2 * (size_t)n * sizeof(double), stream);
    int64_t nl = 0;
    cudaMemsetAsync(w.d_step, 0, 4 * sizeof(int), stream);
    // The step loop is replayed from ONE CUDA graph of kGraphSteps identical launches: the step index lives in device
    // memory, so no launch has step-dependent arguments; launches past the last step return at once.
    constexpr int kGraphSteps = 64;
    const size_t fused_smem = 3 * (size_t)n * sizeof(double);
    // one launch per step while every trailing row still gets its own warp (<= ~16 rows per SM-resident block);
    // beyond that the two-kernel form (one warp per row over a larger grid) is faster (measured: 4096 -> 162 vs 133 ms)
    const bool fused = n <= 3072 && fused_smem <= 200 * 1024 && getenv("VPCA_EIG_TWO_KERNELS") == nullptr;
    const int big_blocks = (n - 1 + 3) / 4 > 0 ? (n - 1 + 3) / 4 : 1;
    if (w.graph_exec == nullptr || w.graph_n != n || w.graph_fused != fused) {
        if (w.graph_exec != nullptr) cudaGraphExecDestroy(w.graph_exec);
        w.graph_exec = nullptr;
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (fused) {
            e = cudaFuncSetAttribute(tridiag_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            if (e != cudaSuccess) return e;
        }
        const int fused_blocks = std::max(1, std::min(sms, (n + 15) / 16));
        cudaGraph_t graph = nullptr;
        e = cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal);
        if (e != cudaSuccess) return e;
        for (int g = 0; g < kGraphSteps; ++g) {
            if (fused) {
                tridiag_fused_kernel<<<fused_blocks, 512, fused_smem, stream>>>(w.d_C, n, w.d_step, w.d_v, w.d_p, w.d_diag,
                                                                                w.d_off, w.d_tau);
            } else {
                tridiag_small_kernel<<<1, kSmallThreads, 0, stream>>>(w.d_C, n, w.d_step, w.d_v, w.d_p, w.d_w, w.d_diag,
                                                                      w.d_off, w.d_tau, w.d_scal);
                tridiag_big_kernel<<<big_blocks, 128, 0, stream>>>(w.d_C, n, w.d_step, w.d_v, w.d_w, w.d_tau, w.d_p);
            }
        }
        e = cudaStreamEndCapture(stream, &graph);
        if (e != cudaSuccess) return e;
        e = cudaGraphInstantiate(&w.graph_exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) return e;
        w.graph_n = n;
        w.graph_fused = fused;
    }
    for (int j = 0; j < n; j += kGraphSteps) {
        e = cudaGraphLaunch(w.graph_exec, stream);
        if (e != cudaSuccess) return e;
        nl += (fused ? 1 : 2) * kGraphSteps;
    }
    bisect_kernel<<<k, 256, 0, stream>>>(w.d_diag, w.d_off, n, w.d_off + n, w.d_evals, w.d_scal);
    const size_t invit_smem = 8 * (size_t)n * sizeof(double);
    if (invit_smem <= 200 * 1024) {
        e = cudaFuncSetAttribute(invit_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;   // (per device: not cached)
        invit_kernel<true><<<1, 256, invit_smem, stream>>>(w.d_diag, w.d_off, n, k, w.d_evals, w.d_scal, w.d_lu,
                                                           w.d_evecs);
    } else {
        invit_kernel<false><<<1, 256, 0, stream>>>(w.d_diag, w.d_off, n, k, w.d_evals, w.d_scal, w.d_lu, w.d_evecs);
    }
    backtransform_kernel<<<k, 512, 0, stream>>>(w.d_C, n, w.d_tau, w.d_evecs);
    nl += 3;
    if (launches) *launches += nl;
    return cudaGetLastError();
}

}  // namespace vpca

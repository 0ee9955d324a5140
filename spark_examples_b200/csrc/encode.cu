// Genotype encode on the device: RDD[Seq[Int]] rows (CSR) -> dense sample-major tile.
//
// Device half of VariantsPcaDriver.getCallsRdd / extractCallInfo
// (reference: src/main/scala/com/google/cloud/genomics/spark/examples/VariantsPca.scala:56-60, :153-168):
// row v lists the callset indices that have `hasVariation` at variant v; the dense equivalent is column v of
// X in {0,1,..}^N where X[s][v] = number of times s is listed (a sample listed twice counts twice, exactly as the
// reference's `for (c1 <- callset; c2 <- callset)` at :187 would count it).  The tile is written sample-major
// (row = sample, contiguous along variants) because that is the K-major operand layout the tcgen05 Gram kernel
// streams through TMA.
//
// Projecting contexts hand a map `rows` (input sample position s -> row rows[s] of the tile; fitted samples first, then
// projected ones): the cells of sample s land in row rows[s], so inputs stay in source order.  rows == nullptr: identity.
//
// HBM-bound scatter: one warp per variant row reads its indices coalesced and adds 1 to X[s][v] with a packed
// 32-bit atomic (4 int8 cells or 2 bf16 cells per word), so duplicates and any index order are handled.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "vpca_internal.h"

namespace vpca {
namespace {

// cell (s, v) of a row-major tile (panel == 0) or of the panel layout (see vpca_internal.h)
__device__ __forceinline__ int64_t cell_index(int s, int64_t v, int64_t ld, int64_t panel, int n) {
    if (panel == 0) return (int64_t)s * ld + v;
    const int64_t pnl = v / panel;
    return pnl * (int64_t)n * panel + (int64_t)s * panel + (v - pnl * panel);
}

template <typename IdxT>
__global__ void encode_i8_kernel(const int64_t* __restrict__ off, int64_t base, const IdxT* __restrict__ idx,
                                 int64_t nv, int n, int max_mult, uint32_t* __restrict__ xw, int64_t ld,
                                 int64_t panel, const int32_t* __restrict__ rows, int* __restrict__ flags) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    int bad = 0;
    for (int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < nv; v += warps) {
        const int64_t e0 = off[v] - base, e1 = off[v + 1] - base;
        for (int64_t e = e0 + lane; e < e1; e += 32) {
            const int s = (int)idx[e];
            if (s < 0 || s >= n) {
                bad |= 1;
                continue;
            }
            const int64_t byte = cell_index(rows != nullptr ? rows[s] : s, v, ld, panel, n);
            const uint32_t shift = (uint32_t)(byte & 3) * 8u;
            const uint32_t old = atomicAdd(xw + (byte >> 2), 1u << shift);
            if ((int)((old >> shift) & 0xFFu) >= max_mult) bad |= 2;
        }
    }
    if (bad) atomicOr(flags, bad);
}

template <typename IdxT>
__global__ void encode_bf16_kernel(const int64_t* __restrict__ off, int64_t base, const IdxT* __restrict__ idx,
                                   int64_t nv, int n, int max_mult, __nv_bfloat162* __restrict__ x2, int64_t ld,
                                   int64_t panel, const int32_t* __restrict__ rows, int* __restrict__ flags) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    int bad = 0;
    for (int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < nv; v += warps) {
        const int64_t e0 = off[v] - base, e1 = off[v + 1] - base;
        for (int64_t e = e0 + lane; e < e1; e += 32) {
            const int s = (int)idx[e];
            if (s < 0 || s >= n) {
                bad |= 1;
                continue;
            }
            const int64_t el = cell_index(rows != nullptr ? rows[s] : s, v, ld, panel, n);
            const bool hi = (el & 1) != 0;
            const __nv_bfloat162 one = __floats2bfloat162_rn(hi ? 0.f : 1.f, hi ? 1.f : 0.f);
            const __nv_bfloat162 old = atomicAdd(x2 + (el >> 1), one);
            const float prev = hi ? __high2float(old) : __low2float(old);
            if (prev >= (float)max_mult) bad |= 2;
        }
    }
    if (bad) atomicOr(flags, bad);
}

// packed e2m1 cells: multiplicity m in {0, 1, 2} is the code 2 m (0b0000, 0b0010 = 1.0, 0b0100 = 2.0), so one
// occurrence adds 2 to the nibble of cell (s, v); eight cells per 32-bit word.
template <typename IdxT>
__global__ void encode_e2m1_kernel(const int64_t* __restrict__ off, int64_t base, const IdxT* __restrict__ idx,
                                   int64_t nv, int n, int max_mult, uint32_t* __restrict__ xw, int64_t ld,
                                   int64_t panel, const int32_t* __restrict__ rows, int* __restrict__ flags) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    int bad = 0;
    for (int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < nv; v += warps) {
        const int64_t e0 = off[v] - base, e1 = off[v + 1] - base;
        for (int64_t e = e0 + lane; e < e1; e += 32) {
            const int s = (int)idx[e];
            if (s < 0 || s >= n) {
                bad |= 1;
                continue;
            }
            const int64_t cell = cell_index(rows != nullptr ? rows[s] : s, v, ld, panel, n);
            const uint32_t shift = (uint32_t)(cell & 7) * 4u;
            const uint32_t old = atomicAdd(xw + (cell >> 3), 2u << shift);
            if ((int)((old >> shift) & 0xFu) >= 2 * max_mult) bad |= 2;
        }
    }
    if (bad) atomicOr(flags, bad);
}

// ---------------------------------------------------------------------------------------------------------------
// Bitmap rows -> cells (SURVEY 8f-1: packed wire format).  Input: one bitmap per variant, bit s (LSB first) of row v =
// sample s has variation; rows `stride` bytes apart.  A warp takes 32 variants x 32 samples: lane = variant loads one
// 32-bit word (32 samples of its variant), 32 ballots transpose the 32 x 32 bit tile so that lane = sample holds the
// 32 variant bits of its sample, which it expands to 32 cells and stores as one contiguous 32-byte (int8) /
// 16-byte (e2m1) / 64-byte (bf16) run of its sample row.  A bit-matrix transpose at HBM speed; no atomics.
// CODE 0: rows are bitmaps (1 bit per sample).  CODE 1 / 2: rows are PLINK .bed rows (2 bits per sample, low bits
// first; 00 hom A1, 01 missing, 10 het, 11 hom A2) and the carrier bit is "has an A1" (codes 00, 10 = low bit clear) /
// "has an A2" (codes 10, 11 = high bit set); a missing call carries nothing, like a no-call under VariantsPca.scala:58.
__device__ __forceinline__ uint32_t compress_even_bits(uint64_t x) {   // bit 2j of x -> bit j
    x &= 0x5555555555555555ull;
    x = (x | (x >> 1)) & 0x3333333333333333ull;
    x = (x | (x >> 2)) & 0x0F0F0F0F0F0F0F0Full;
    x = (x | (x >> 4)) & 0x00FF00FF00FF00FFull;
    x = (x | (x >> 8)) & 0x0000FFFF0000FFFFull;
    x = (x | (x >> 16)) & 0x00000000FFFFFFFFull;
    return (uint32_t)x;
}

template <int BITS>
__global__ void bits_to_cells_kernel(const uint8_t* __restrict__ bits, int64_t stride, int64_t nv, int n,
                                     uint8_t* __restrict__ x, int64_t ld, int64_t panel, int code,
                                     const int32_t* __restrict__ rows) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int words = (n + 31) / 32;                          // 32-sample words per variant
    const int64_t vgroups = (nv + 31) / 32;
    if (warp >= vgroups * words) return;
    const int64_t vg = warp / words;
    const int k = (int)(warp - vg * words);
    const int64_t v = vg * 32 + lane;                         // my variant while loading
    uint32_t word = 0;
    if (v < nv && code == 0) {
        const uint8_t* row = bits + v * stride + (size_t)k * 4;
        const int64_t avail = stride - (int64_t)k * 4;        // bytes of this row from here on
#pragma unroll
        for (int b = 0; b < 4; ++b)
            if (b < avail) word |= (uint32_t)row[b] << (8 * b);
    } else if (v < nv) {
        const uint8_t* row = bits + v * stride + (size_t)k * 8;   // 32 samples = 8 bytes of 2-bit codes
        const int64_t avail = stride - (int64_t)k * 8;
        uint64_t w = 0;
#pragma unroll
        for (int b = 0; b < 8; ++b)
            if (b < avail) w |= (uint64_t)row[b] << (8 * b);
        // padding samples (code 00 = "hom A1") beyond n are masked below (smp >= n)
        word = code == 1 ? ~compress_even_bits(w) : compress_even_bits(w >> 1);
    }
    uint32_t mine = 0;                                        // after the loop: bit j = variant vg*32+j at MY sample
#pragma unroll
    for (int b = 0; b < 32; ++b) {
        const uint32_t m = __ballot_sync(0xffffffffu, (word >> b) & 1u);
        if (lane == b) mine = m;
    }
    const int smp = k * 32 + lane;
    if (smp >= n) return;
    const int64_t v0 = vg * 32;
    const int row = rows != nullptr ? rows[smp] : smp;
    // cell index of (row, v0): 32 consecutive cells never straddle a panel (panels are multiples of 128 cells)
    int64_t cell;
    if (panel == 0) cell = (int64_t)row * ld + v0;
    else {
        const int64_t pnl = v0 / panel;
        cell = pnl * (int64_t)n * panel + (int64_t)row * panel + (v0 - pnl * panel);
    }
    if constexpr (BITS == 8) {
        uint32_t o[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const uint32_t nib = (mine >> (4 * q)) & 0xFu;
            o[q] = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
        }
        uint4* dst = reinterpret_cast<uint4*>(x + cell);
        dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
        dst[1] = make_uint4(o[4], o[5], o[6], o[7]);
    } else if constexpr (BITS == 4) {
        uint32_t o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint32_t byte = (mine >> (8 * q)) & 0xFFu;   // 8 variants -> 8 nibbles, carrier = code 2
            uint32_t w = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) w |= ((byte >> i) & 1u) << (4 * i + 1);
            o[q] = w;
        }
        *reinterpret_cast<uint4*>(x + cell / 2) = make_uint4(o[0], o[1], o[2], o[3]);
    } else {
        uint32_t o[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const uint32_t two = (mine >> (2 * q)) & 3u;       // bf16 1.0 = 0x3F80
            o[q] = ((two & 1u) ? 0x3F80u : 0u) | ((two & 2u) ? 0x3F800000u : 0u);
        }
        uint4* dst = reinterpret_cast<uint4*>(x + cell * 2);
#pragma unroll
        for (int q = 0; q < 4; ++q) dst[q] = make_uint4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
    }
}

}  // namespace

cudaError_t encode_bits(const uint8_t* d_bits, int64_t stride, int64_t nv, int n, int elem_bits, void* d_x, int64_t ld,
                        int64_t panel, int code, const int32_t* d_rows, cudaStream_t stream) {
    if (nv <= 0) return cudaSuccess;
    // every cell of the touched 32-variant groups is written, so only a partial last panel / k-block needs zeroing
    cudaError_t e = cudaSuccess;
    if (panel > 0) {
        const int64_t npanels = (nv + panel - 1) / panel;
        if (npanels * panel != ((nv + 31) / 32) * 32)
            e = cudaMemsetAsync(static_cast<char*>(d_x) + (size_t)(npanels - 1) * n * panel * elem_bits / 8, 0,
                                (size_t)n * panel * elem_bits / 8, stream);
    } else {
        const size_t pitch = (size_t)ld * elem_bits / 8;
        size_t width = (((size_t)nv + 127) / 128) * 128 * elem_bits / 8;
        if (width > pitch) width = pitch;
        e = cudaMemset2DAsync(d_x, pitch, 0, width, (size_t)n, stream);
    }
    if (e != cudaSuccess) return e;
    const int64_t warps = ((nv + 31) / 32) * ((n + 31) / 32);
    const int threads = 256;
    const int64_t blocks = (warps * 32 + threads - 1) / threads;
    if (elem_bits == 8)
        bits_to_cells_kernel<8><<<(unsigned)blocks, threads, 0, stream>>>(d_bits, stride, nv, n, static_cast<uint8_t*>(d_x), ld, panel, code,
                                                                          d_rows);
    else if (elem_bits == 4)
        bits_to_cells_kernel<4><<<(unsigned)blocks, threads, 0, stream>>>(d_bits, stride, nv, n, static_cast<uint8_t*>(d_x), ld, panel, code,
                                                                          d_rows);
    else
        bits_to_cells_kernel<16><<<(unsigned)blocks, threads, 0, stream>>>(d_bits, stride, nv, n, static_cast<uint8_t*>(d_x), ld, panel, code,
                                                                          d_rows);
    return cudaGetLastError();
}

template <typename IdxT>
static cudaError_t encode_launch(const int64_t* d_off, int64_t base, const IdxT* d_idx, int64_t nv, int n, int elem_bits,
                                 int max_mult, void* d_x, int64_t ld, int64_t panel, const int32_t* d_rows, int* d_flags,
                                 cudaStream_t stream);

cudaError_t encode_calls(const int64_t* d_off, int64_t base, const void* d_idx, int idx_bytes, int64_t nv, int n,
                         int elem_bits, int max_mult, void* d_x, int64_t ld, int64_t panel, const int32_t* d_rows,
                         int* d_flags, cudaStream_t stream) {
    if (idx_bytes == 2)
        return encode_launch(d_off, base, static_cast<const uint16_t*>(d_idx), nv, n, elem_bits, max_mult, d_x, ld, panel,
                             d_rows, d_flags, stream);
    return encode_launch(d_off, base, static_cast<const int32_t*>(d_idx), nv, n, elem_bits, max_mult, d_x, ld, panel, d_rows,
                         d_flags, stream);
}

template <typename IdxT>
static cudaError_t encode_launch(const int64_t* d_off, int64_t base, const IdxT* d_idx, int64_t nv, int n, int elem_bits,
                                 int max_mult, void* d_x, int64_t ld, int64_t panel, const int32_t* d_rows, int* d_flags,
                                 cudaStream_t stream) {
    cudaError_t e = cudaSuccess;
    if (panel > 0) {
        // whole panels are contiguous: zero every panel the rows touch
        const size_t npanels = (size_t)((nv + panel - 1) / panel);
        if (npanels > 0) e = cudaMemsetAsync(d_x, 0, npanels * (size_t)n * (size_t)panel * elem_bits / 8, stream);
    } else {
        // zero the nv columns (rounded up to the k-block of 128 cells / 128 bytes the Gram kernel reads) of every row
        const size_t pitch = (size_t)ld * elem_bits / 8;
        size_t width = elem_bits == 4 ? (((size_t)nv + 127) / 128) * 64 : ((((size_t)nv * elem_bits / 8) + 127) / 128) * 128;
        if (width > pitch) width = pitch;
        if (width > 0) e = cudaMemset2DAsync(d_x, pitch, 0, width, (size_t)n, stream);
    }
    if (e != cudaSuccess || nv <= 0) return e;
    const int threads = 256;
    const int64_t want = (nv * 32 + threads - 1) / threads;
    const int blocks = (int)(want < 148 * 16 ? (want < 1 ? 1 : want) : 148 * 16);
    if (elem_bits == 4) {
        const int cap = max_mult > 2 ? 2 : max_mult;
        encode_e2m1_kernel<IdxT><<<blocks, threads, 0, stream>>>(d_off, base, d_idx, nv, n, cap, reinterpret_cast<uint32_t*>(d_x),
                                                           ld, panel, d_rows, d_flags);
    } else if (elem_bits == 8) {
        const int cap = max_mult > 127 ? 127 : max_mult;
        encode_i8_kernel<IdxT><<<blocks, threads, 0, stream>>>(d_off, base, d_idx, nv, n, cap, reinterpret_cast<uint32_t*>(d_x), ld,
                                                         panel, d_rows, d_flags);
    } else {
        const int cap = max_mult > 256 ? 256 : max_mult;   // bf16 holds integers exactly up to 256
        encode_bf16_kernel<IdxT><<<blocks, threads, 0, stream>>>(d_off, base, d_idx, nv, n, cap,
                                                           reinterpret_cast<__nv_bfloat162*>(d_x), ld, panel, d_rows, d_flags);
    }
    return cudaGetLastError();
}

// Loads the encode kernels on the current device (see gram_preload_kernels: a first launch must never be the thing a host
// thread blocks on while a peer barrier of the same process is spinning).
cudaError_t encode_preload_kernels() {
    cudaFuncAttributes fa;
    cudaError_t e = cudaSuccess;
#define VPCA_LOAD(k) if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, k)
    VPCA_LOAD((encode_i8_kernel<int32_t>)); VPCA_LOAD((encode_i8_kernel<uint16_t>));
    VPCA_LOAD((encode_bf16_kernel<int32_t>)); VPCA_LOAD((encode_bf16_kernel<uint16_t>));
    VPCA_LOAD((encode_e2m1_kernel<int32_t>)); VPCA_LOAD((encode_e2m1_kernel<uint16_t>));
    VPCA_LOAD((bits_to_cells_kernel<8>)); VPCA_LOAD((bits_to_cells_kernel<4>)); VPCA_LOAD((bits_to_cells_kernel<16>));
#undef VPCA_LOAD
    return e;
}

}  // namespace vpca

// Gram / similarity accumulation  S += X X^T  on sm_100a tensor cores.
//
// Replaces the hot loop of VariantsPcaDriver.getSimilarityMatrix
// (reference: src/main/scala/com/google/cloud/genomics/spark/examples/VariantsPca.scala:182-191,
//  `for (c1 <- callset; c2 <- callset) matrix(c1, c2) += 1` over every variant) by a dense symmetric
// rank-V update on the genotype matrix X (samples x variants, sample-major in HBM):
//
//   TMA (cp.async.bulk.tensor, SWIZZLE_128B)  ->  shared memory ring  ->  tcgen05.mma (kind::i8 / kind::f16)
//   ->  int32 / fp32 accumulators in TMEM  ->  tcgen05.ld  ->  red.global.add.s32 into the lower triangle of S.
//
// Work decomposition ("window-synchronous stream-K"):
//   * an output tile is the product of A row blocks (128 samples each: one per CTA, so two with cta_group::2) and up to
//     256 B rows; its accumulator holds D[m][n] = sum_v X[rowA + m][v] * X[rowB + n][v] and is written TRANSPOSED,
//     S[rowB + n][rowA + m], so that the 32 lanes of a warp (= 32 consecutive m) hit 32 consecutive int32 of one row of S;
//   * default tiling: rectangles of 256 A rows (two adjacent 128-blocks) x up to 256 B rows that touch row >= col, the B
//     strips of nearly equal width (2504 samples: 7 x 256 + 3 x 240; kind::mxf4: 3 x 240 + 8 x 224 because its block scales
//     take 16 TMEM columns), so that tiles have nearly equal weight and a worker never spans three of them;
//   * EXACT BLOCK COVER (VPCA_EXACT_COVER=1; int8 / bf16 / f8f6f4; measured SLOWER on B200 and therefore off by default --
//     its N = 128 tiles need 96 B/clk per SM from L2 where a 256 x 256 tile needs 64, and L2 -> SM delivers ~58): in units
//     of 128 x 128 blocks the lower triangle of S has nb (nb + 1) / 2 blocks, and a tile always multiplies TWO A blocks
//     (M = 256: an MMA costs 128 rows per CTA whatever it needs), so the square tiling pays 4 blocks for each of the nb / 2
//     diagonal tiles although only 3 are needed.  The A blocks of a pair need not be adjacent and the B rows may be a
//     single block (N = 128), and a block above the diagonal may be computed in place of its mirror image and written
//     transposed; with that freedom the tile list of build_tiles covers every needed block exactly once (2504 samples:
//     210 blocks instead of 220, 4.5 % less MMA work);
//   * owner-computes bands: a context that stores only rows [own_lo, own_hi) of S and has no peers enumerates only the
//     tiles of those rows (every variant is fed to every band's context; nothing is flushed anywhere else);
//   * projecting contexts: X has N + M rows (fitted, then projected samples) and S has N columns at pitch N; the B strips
//     run over all N + M rows, the A blocks over the N fitted ones, so rows N.. of S are the M x N cross block;
//   * the variant axis is cut into k-blocks of 128 bytes (one swizzle atom) and into windows of `kb_window`
//     k-blocks; in every window the (tile, k-block) units are split evenly over the workers (CTA pairs), and all
//     workers walk the windows in the same order, so the slice of X a window needs (n x kb_window*128 B, sized to
//     sit in L2) is fetched from HBM once and re-read from L2 by the other tiles;
//   * when the pieces of every worker fit its TMEM columns (N = 2504: 55 tiles, 74 pairs: a worker touches <= 2 tiles,
//     always the same ones) the accumulators stay resident in TMEM for the whole launch and are flushed once at the end;
//     otherwise (large N) it is whole-tile waves + a stream-K tail with double-buffered accumulators;
//   * the split of a window over the workers is speed-weighted from launch to launch (rebalance_kernel, repair_split);
//   * the flush packs two cells into one 64-bit red (no carry between the halves: counts are non-negative, sums < 2^31).
// Integer atomics make the result independent of the order of the flushes: S is bit-exact.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstring>

#include <algorithm>
#include <map>
#include <mutex>
#include <tuple>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "ptx_sm100.cuh"
#include "vpca_internal.h"

namespace vpca {

namespace {

constexpr int kThreads = 256;
constexpr int kKBytes = 128;                    // bytes of K per k-block: one SWIZZLE_128B atom
constexpr int kBoxRows = 128;                   // rows per TMA box
constexpr int kBoxBytes = kBoxRows * kKBytes;   // 16 KiB
constexpr int kUmmaN = 256;
constexpr int kUmmaNScaled = 240;               // kind::mxf4: 2 x 240 accumulator columns + 16 scale-factor columns
constexpr uint32_t kSfCol = 480;                // TMEM column of the (constant 1.0) block scale factors
constexpr uint32_t kTmemCols = 512;             // two 256-column accumulators
constexpr long long kWatchdogCycles = 20000000000LL;   // ~10 s: a stuck barrier traps instead of hanging the box

template <int CG, int KIND = 0>
struct Cfg {
    static constexpr int A_BYTES = kBoxBytes;                  // per CTA per stage
    static constexpr int B_BYTES = (kUmmaN / CG) * kKBytes;    // per CTA per stage (32 KiB / 16 KiB): whole 128-row boxes
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int STAGES = CG == 1 ? 4 : 6;
    static constexpr int BAR_BYTES = 256;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + BAR_BYTES + 1024;   // + slack for 1024 B alignment
};

constexpr int kMaxPeers = 16;

// One output tile: (A block of CTA 0, A block of CTA 1) x (n_eff B rows from rowB).
struct TileDesc {
    int rowA0, rowA1;   // first sample of the A block of CTA 0 / CTA 1 (cta_group::1: rowA0 only)
    int rowB;           // first sample of the B rows
    int n_eff;          // MMA N: B rows that exist, rounded up to 16
    int wstart;         // sum of the weights (n_eff / 16) of the tiles before this one
    int flags;          // kTileXpose: a 128-block above the diagonal is written transposed (it stands in for its mirror
                        // image) instead of being skipped; kTileFiller: CTA 1's A block only pads the pair, drop its output
    int acc_cols;       // TMEM columns its accumulator takes: n_eff rounded up to 32 (exact cover), else the tiling's BN
                        // (256, or 240 for kind::mxf4 whose two accumulators sit below the scale columns at 480)
    int pad1;
};
constexpr int kTileXpose = 1, kTileFiller = 2, kTileSelfB = 4;   // kTileSelfB: the B rows ARE the pair's two A blocks (a
                                                                  // diagonal 256 x 256 tile): B is read from the A tile, no B load
constexpr int kMaxSegs = 4;   // (tile, k-range) pieces one worker may own per window in resident mode

struct GramArgs {
    int32_t* S;
    int32_t* peer[kMaxPeers];   // num_peers > 0: the flush goes to peer-mapped Grams (own included) over NVLink:
    int num_peers;              //   peer_mode 0: into ALL of them (replicated reduce);
    int peer_mode;              //   peer_mode 1: only into the Gram of the rank that owns the row (reduce-scatter)
    int own_end[kMaxPeers];     // rank q owns Gram rows [own_end[q-1], own_end[q]); multiples of 32, >= 32 apart
    const TileDesc* tiles;
    int* err;          // mapped host memory: watchdog diagnostics
    int n_cols;        // columns of S, also its row pitch: the fitted samples.  X may have more rows (projected samples,
                       // rows n_cols .. row_limit - 1 of S); A blocks reaching past n_cols read them, and the guard
                       // col < n_cols keeps those products out of S (at pitch n_cols they would land in the next row)
    int num_tiles;
    int num_full;      // leading tiles of full weight: what the large-N schedule deals out in whole-tile waves
    int total_weight;  // sum of n_eff / 16 over all tiles
    int kb_total;
    int kb_window;
    int num_workers;
    int resident;
    int elems_per_kb;  // 128 / sizeof(element)
    int kb_per_panel;  // k-blocks per panel of the genotype matrix (row-major input = one panel)
    int sync_lead;     // > 0: a worker may run at most this many windows ahead of the slowest one (soft barrier)
    int active_workers;
    int* win_done;     // win_done[w] = number of workers whose producer has issued every load of window w
    long long* prof;   // optional per-CTA timestamps (globaltimer ns): start, first MMA, MMA done, end
    const double* cum; // cum[w] = fraction of every window's units owned by workers < w (cum[0] = 0, cum[W] = 1)
    int col_limit;     // TMEM columns the accumulators of one worker may take (512; mxf4: 480)
    int acc_stride;    // large-N schedule: TMEM columns between the two double-buffered accumulators (256; mxf4: 240)
    int row_limit;     // rows of S at or beyond this one are never written (n, or the end of an owner-computes band)
    int red64;         // epilogue packs two cells per 64-bit red (VPCA_RED64=0: one 32-bit red per cell)
    int tx_shift;      // TMA transaction bytes per stage = STAGE_BYTES >> tx_shift (1 for packed 4-bit sources: the
                       // mbarrier counts the 8 data bytes of every 16-byte shared-memory chunk, not the gap)
};

struct Seg {
    int tile, kb0, kb1, col, slot, first, flush, use, win, last_in_win;   // slot: which accumulator barrier pair
    int rowA0, rowA1, rowB, n_eff, flags;
};

// The pieces of a weighted unit range [u_begin, u_end) -- tile t occupies [wstart_t * len, (wstart_t + w_t) * len) and its
// k-block q sits at wstart_t * len + q * w_t -- as (tile, k-range, TMEM column) triples.  Two workers that share a
// boundary u agree on the k-block it falls in (both take floor((u - base) / w_t)), so the pieces partition every tile.
// Shared by the kernel, by the host (which decides whether the accumulators of a worker fit TMEM) and by the rebalancer.
struct SegPlan {
    int n;
    int tile[kMaxSegs], lo[kMaxSegs], hi[kMaxSegs], col[kMaxSegs];
    int cols;      // TMEM columns needed
    int overflow;  // more than kMaxSegs pieces
};

__host__ __device__ inline void plan_segments(const TileDesc* tiles, int num_tiles, int first_tile, long long u_begin,
                                              long long u_end, int len, SegPlan& p) {
    p.n = 0;
    p.cols = 0;
    p.overflow = 0;
    const long long origin = (long long)tiles[first_tile].wstart * len;
    long long u = u_begin;
    int t = first_tile;
    while (u < u_end && t < num_tiles) {
        const int w = tiles[t].n_eff >> 4;
        const long long base = (long long)tiles[t].wstart * len - origin;
        const long long tend = base + (long long)w * len;
        if (tend <= u) {
            ++t;
            continue;
        }
        const long long e = u_end < tend ? u_end : tend;
        const int lo = (int)((u - base) / w);
        const int hi = e == tend ? len : (int)((e - base) / w);
        u = e;
        if (lo >= hi) continue;   // a sliver thinner than one k-block: the neighbour owns that k-block
        if (p.n == kMaxSegs) {
            p.overflow = 1;
            return;
        }
        p.tile[p.n] = t;
        p.lo[p.n] = lo;
        p.hi[p.n] = hi;
        p.col[p.n] = p.cols;
        p.cols += tiles[t].acc_cols;
        ++p.n;
    }
}

// Largest e <= u_end such that the pieces of [u_begin, e) fit one worker's TMEM (at most kMaxSegs accumulators,
// at most col_limit columns): u_end itself, or the start of the first tile whose accumulator no longer fits.
// `hint`: a tile index at or before the tile that holds u_begin (advanced to it; callers walk u_begin upwards).
__host__ __device__ inline long long feasible_end(const TileDesc* tiles, int num_tiles, long long u_begin, long long u_end,
                                                  int len, int col_limit, int& hint) {
    int n = 0, cols = 0;
    long long u = u_begin;
    int t = hint;
    bool first = true;
    while (u < u_end && t < num_tiles) {
        const int w = tiles[t].n_eff >> 4;
        const long long base = (long long)tiles[t].wstart * len;
        const long long tend = base + (long long)w * len;
        if (tend <= u) {
            ++t;
            continue;
        }
        if (first) {
            hint = t;
            first = false;
        }
        const long long e = u_end < tend ? u_end : tend;
        const int lo = (int)((u - base) / w);
        const int hi = e == tend ? len : (int)((e - base) / w);
        if (lo < hi) {
            if (n == kMaxSegs || cols + tiles[t].acc_cols > col_limit) return u;
            ++n;
            cols += tiles[t].acc_cols;
        }
        u = e;
    }
    return u_end;
}

// Makes a candidate split (cand[0] = 0 <= cand[1] <= ... <= cand[workers] = 1, fractions of the uw units of a window)
// feasible: worker i ends where feasible_end says it must, and worker i + 1 starts there.  False if the last worker
// cannot reach the end of the window (the caller keeps the old split).
__host__ __device__ inline bool repair_split(const TileDesc* tiles, int num_tiles, int workers, long long uw, int len,
                                             int col_limit, double* cand) {
    long long ub = 0;
    int hint = 0;
    for (int i = 0; i < workers; ++i) {
        long long ue = (i + 1 == workers) ? uw : (long long)((double)uw * cand[i + 1]);
        if (ue < ub) ue = ub;
        const long long fe = feasible_end(tiles, num_tiles, ub, ue, len, col_limit, hint);
        if (fe < ue) {
            if (i + 1 == workers) return false;
            ue = fe;
        }
        if (i + 1 < workers) cand[i + 1] = ((double)ue + 0.5) / (double)uw;   // floor(uw * cand) == ue in the kernel
        ub = ue;
    }
    return true;
}

// Every role of a worker (TMA producer, MMA issuer, epilogue) replays the same deterministic schedule.
//   resident (every worker's accumulators fit TMEM):  window-synchronous stream-K -- the worker owns the same pieces
//               (tile, k-range) in every window, so its accumulators stay in TMEM for the whole launch;
//   otherwise:  full tiles in waves (wave i = tiles [i W, (i+1) W), one per worker, whole K) -- the tile list is ordered
//               so that a wave is a compact 2-D block of S and shares few row panels of X -- then the leftover
//               tiles are split stream-K style over all workers; accumulators double-buffered against the epilogue.
struct Sched {
    SegPlan plan;
    long long u_begin, u_end, u;
    int kbw, nwin, kb_total, resident, win, seg_i, nflush, acc_stride;
    int worker, workers, num_tiles, wave, full_waves, tail_first;
    const TileDesc* tiles;

    __device__ void init(const GramArgs& a, int w) {
        kbw = a.kb_window;
        kb_total = a.kb_total;
        resident = a.resident;
        acc_stride = a.acc_stride;
        worker = w;
        workers = a.num_workers;
        num_tiles = a.num_tiles;
        tiles = a.tiles;
        nwin = (kb_total + kbw - 1) / kbw;
        win = 0;
        seg_i = 0;
        nflush = 0;
        wave = 0;
        if (resident) {
            const long long uw = (long long)a.total_weight * kbw;
            // speed-weighted split (equal shares until the first launches have been timed, see rebalance_kernel)
            u_begin = (long long)((double)uw * a.cum[worker]);
            u_end = (worker + 1 == a.num_workers) ? uw : (long long)((double)uw * a.cum[worker + 1]);
            plan_segments(tiles, num_tiles, 0, u_begin, u_end, kbw, plan);
            if (plan.overflow || plan.cols > a.col_limit) {   // overlapping accumulators would corrupt S silently
                if (a.err != nullptr && threadIdx.x == 0) {
                    a.err[0] = 9;
                    a.err[1] = (int)blockIdx.x;
                    a.err[2] = plan.cols;
                    a.err[3] = plan.n;
                    __threadfence_system();
                }
                __trap();
            }
        } else {
            full_waves = a.num_full / workers;
            tail_first = full_waves * workers;
            const long long tail_units =
                tail_first < num_tiles ? (long long)(a.total_weight - tiles[tail_first].wstart) * kb_total : 0;
            u_begin = tail_units * worker / workers;       // weighted units of the leftover tiles
            u_end = tail_units * (worker + 1) / workers;
            plan.n = 0;
        }
        u = u_begin;
    }
    __device__ void fill(Seg& s, int t) const {
        const int4 lo = __ldg(reinterpret_cast<const int4*>(tiles + t));
        const int4 hi = __ldg(reinterpret_cast<const int4*>(tiles + t) + 1);
        s.tile = t;
        s.rowA0 = lo.x;
        s.rowA1 = lo.y;
        s.rowB = lo.z;
        s.n_eff = lo.w;
        s.flags = hi.y;
    }
    __device__ bool next(Seg& s) {
        if (!resident) {
            s.win = 0;
            s.last_in_win = 0;
            s.first = 1;
            s.flush = 1;
            s.slot = nflush & 1;
            s.col = s.slot * acc_stride;
            s.use = nflush >> 1;
            if (wave < full_waves) {                        // one whole tile of the current wave
                fill(s, wave * workers + worker);
                s.kb0 = 0;
                s.kb1 = kb_total;
                ++wave;
                ++nflush;
                return true;
            }
            // stream-K tail: at most kMaxSegs pieces are planned at a time
            while (true) {
                if (seg_i < plan.n) {
                    fill(s, plan.tile[seg_i]);
                    s.kb0 = plan.lo[seg_i];
                    s.kb1 = plan.hi[seg_i];
                    ++seg_i;
                    ++nflush;
                    return true;
                }
                if (u >= u_end) return false;
                // plan the next pieces: advance u to the end of what was planned
                plan_segments(tiles, num_tiles, tail_first, u, u_end, kb_total, plan);
                seg_i = 0;
                if (plan.n == 0) return false;
                const int lt = plan.tile[plan.n - 1];
                const long long base = (long long)(tiles[lt].wstart - tiles[tail_first].wstart) * kb_total;
                const long long endu = base + (long long)plan.hi[plan.n - 1] * (tiles[lt].n_eff >> 4);
                u = plan.overflow ? endu : u_end;
            }
        }
        if (plan.n == 0) return false;
        if (seg_i == plan.n) {
            ++win;
            seg_i = 0;
        }
        if (win >= nwin) return false;
        const int i = seg_i++;
        fill(s, plan.tile[i]);
        const int base = win * kbw;
        const int cnt = min(kbw, kb_total - base);
        s.kb0 = base + min(plan.lo[i], cnt);
        s.kb1 = base + min(plan.hi[i], cnt);
        s.win = win;
        s.last_in_win = (seg_i == plan.n);
        s.col = plan.col[i];
        s.slot = i;
        s.first = (win == 0);
        s.flush = (win == nwin - 1);
        s.use = 0;
        return true;
    }
};

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err, int code) {
    if (ptx::mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!ptx::mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > kWatchdogCycles) {
            if (err != nullptr) {
                err[0] = code;
                err[1] = (int)blockIdx.x;
                err[2] = (int)bar;
                err[3] = (int)parity;
                __threadfence_system();
            }
            __trap();
        }
    }
}

__device__ __forceinline__ long long globaltimer_ns() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Soft inter-worker barrier: wait (bounded) until `need` workers have finished issuing window `w`.  Purely a pacing
// hint that keeps all workers inside the same few L2-resident windows of X; correctness never depends on it.
__device__ __forceinline__ void wait_window(const int* win_done, int w, int need) {
    const long long t0 = globaltimer_ns();
    while (true) {
        int v;
        asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(win_done + w) : "memory");
        if (v >= need) return;
        if (globaltimer_ns() - t0 > 200000) return;   // 200 us: give up (e.g. not all workers co-resident)
        __nanosleep(256);
    }
}

// K-major SWIZZLE_128B operand tile: rows of 128 B, 8-row groups 1024 B apart (SBO), one atom along K (LBO unused).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

template <int CG, int KIND>
__device__ __forceinline__ uint32_t make_instr_desc(uint32_t N) {
    constexpr uint32_t M = 128 * CG;
    // c_format [4,6): 1 = F32, 2 = S32; a/b_format [7,10)/[10,13): kind::i8 -> 1 (signed int8), kind::f16 -> 1 (BF16),
    // kind::f8f6f4 -> 5 (E2M1); a/b major bits 15/16 = 0 (K-major); n_dim [17,23) = N >> 3; m_dim [24,29) = M >> 4.
    if constexpr (KIND == 3) {
        // block-scaled descriptor (kind::mxf4): a/b_format 1 = E2M1, bit 23 scale_format 1 = UE8M0, sf ids 0, K = 64
        return (1u << 7) | (1u << 10) | ((N >> 3) << 17) | (1u << 23) | ((M >> 4) << 24);
    }
    constexpr uint32_t cfmt = (KIND == 0) ? 2u : 1u;
    constexpr uint32_t abfmt = (KIND == 2) ? 5u : 1u;
    return (cfmt << 4) | (abfmt << 7) | (abfmt << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

template <int CG, int KIND>
__global__ void __launch_bounds__(kThreads, 1) gram_kernel(const __grid_constant__ CUtensorMap tmap,
                                                           const __grid_constant__ CUtensorMap tmap_half, const GramArgs a) {
    using C = Cfg<CG, KIND>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const uint32_t smem_base = ptx::smem_u32(smem);
    const uint32_t bar_base = smem_base + C::STAGES * C::STAGE_BYTES;
    auto sA = [&](uint32_t st) { return smem_base + st * C::A_BYTES; };
    auto sB = [&](uint32_t st) { return smem_base + C::STAGES * C::A_BYTES + st * C::B_BYTES; };
    auto full_bar = [&](uint32_t i) { return bar_base + 8u * i; };
    auto empty_bar = [&](uint32_t i) { return bar_base + 8u * (C::STAGES + i); };
    // accumulator barriers: resident schedule -- one "full" barrier per accumulator of the worker (each completes once);
    // large-N schedule -- two accumulators double-buffered through full / empty pairs 0 and 1
    auto tfull_bar = [&](uint32_t i) { return bar_base + 8u * (2 * C::STAGES + i); };
    auto tempty_bar = [&](uint32_t i) { return bar_base + 8u * (2 * C::STAGES + kMaxSegs + i); };
    volatile uint32_t* tmem_ptr_smem =
        reinterpret_cast<volatile uint32_t*>(smem + C::STAGES * C::STAGE_BYTES + 8 * (2 * C::STAGES + kMaxSegs + 2));

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const uint32_t lane = ptx::lane_id();
    const uint32_t cta_rank = (CG == 2) ? ptx::cluster_ctarank() : 0u;
    const bool leader = cta_rank == 0;
    const int worker = (CG == 2) ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const bool issuer = ptx::elect_one();   // one fixed lane per warp issues TMA / MMA / commits

    if constexpr (CG == 2) ptx::cluster_sync();   // both CTAs of the pair are resident before the paired TMEM alloc

    if (warp == 0 && issuer) {
        ptx::prefetch_tensormap(&tmap);
        ptx::prefetch_tensormap(&tmap_half);
    } else if (warp == 1 && issuer) {
        for (uint32_t i = 0; i < (uint32_t)C::STAGES; ++i) {
            ptx::mbar_init(full_bar(i), CG);    // producer arrive(s): leader expect_tx (+ peer's remote arrive)
            ptx::mbar_init(empty_bar(i), 1);    // one tcgen05.commit per use
        }
        for (uint32_t i = 0; i < (uint32_t)kMaxSegs; ++i) ptx::mbar_init(tfull_bar(i), 1);
        for (uint32_t i = 0; i < 2; ++i) ptx::mbar_init(tempty_bar(i), CG * 128);   // every epilogue thread of the pair arrives at the leader
        ptx::fence_mbar_init();
    } else if (warp == 2) {
        ptx::tmem_alloc<CG>(ptx::smem_u32(const_cast<uint32_t*>(tmem_ptr_smem)), kTmemCols);
        ptx::tmem_relinquish<CG>();
    }
    ptx::tc_fence_before();
    if constexpr (CG == 2) ptx::cluster_sync(); else __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;
    if constexpr (KIND == 3) {
        // kind::mxf4 multiplies every 32-cell block by a UE8M0 scale read from TMEM; genotype cells are unscaled, so
        // the 16 scale columns of both CTAs are filled once with 0x7F = 2^0 (any scale-factor id / layout reads 1.0).
        if (warp >= 4) {
            ptx::tmem_st_32x32b_x16_const(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + kSfCol, 0x7F7F7F7Fu);
            ptx::tmem_st_wait();
        }
        ptx::tc_fence_before();
        if constexpr (CG == 2) ptx::cluster_sync(); else __syncthreads();
        ptx::tc_fence_after();
    }
    if (a.prof != nullptr && threadIdx.x == 0) a.prof[(size_t)blockIdx.x * 4 + 0] = globaltimer_ns();

    if (warp == 0) {
        // ===================================== TMA producer =====================================
        if (issuer) {
            Sched sc;
            sc.init(a, worker);
            Seg s;
            uint32_t it = 0;
            int synced_win = -1;
            while (sc.next(s)) {
                // with cta_group::2 each CTA supplies its own A block and half of the N = n_eff B rows
                const int rowA = (CG == 2 && cta_rank != 0) ? s.rowA1 : s.rowA0;
                const int rowB = s.rowB + ((CG == 2) ? (int)cta_rank * (s.n_eff / 2) : 0);
                // B rows per CTA: a 64-row box is enough for the N <= 128 tiles of the exact block cover (cta_group::2)
                const bool half_box = (CG == 2) && (s.n_eff <= 128);
                const bool two_boxes = (CG == 1) && (s.n_eff > kBoxRows);
                const bool self_b = (CG == 2) && (s.flags & kTileSelfB) != 0;   // B = the A blocks themselves: nothing to load
                const uint32_t tx_cta =
                    (uint32_t)(C::A_BYTES + (self_b ? 0 : (half_box ? kBoxBytes / 2 : (two_boxes ? 2 * kBoxBytes : kBoxBytes))));
                if (a.sync_lead > 0 && leader && s.win != synced_win) {
                    synced_win = s.win;
                    if (s.win >= a.sync_lead) wait_window(a.win_done, s.win - a.sync_lead, a.active_workers);
                }
                for (int kb = s.kb0; kb < s.kb1; ++kb, ++it) {
                    const uint32_t st = it % C::STAGES, ph = (it / C::STAGES) & 1u;
                    mbar_wait(empty_bar(st), ph ^ 1u, a.err, 1);
                    const int pnl = kb / a.kb_per_panel;
                    const int kc = (kb - pnl * a.kb_per_panel) * a.elems_per_kb;
                    if constexpr (CG == 1) {
                        ptx::mbar_arrive_expect_tx(full_bar(st), tx_cta >> a.tx_shift);
                        ptx::tma_load_3d(sA(st), &tmap, full_bar(st), kc, rowA, pnl);
                        ptx::tma_load_3d(sB(st), &tmap, full_bar(st), kc, rowB, pnl);
                        if (two_boxes) ptx::tma_load_3d(sB(st) + kBoxBytes, &tmap, full_bar(st), kc, rowB + kBoxRows, pnl);
                    } else {
                        ptx::tma_load_3d_2sm(sA(st), &tmap, full_bar(st), kc, rowA, pnl);
                        if (!self_b) ptx::tma_load_3d_2sm(sB(st), half_box ? &tmap_half : &tmap, full_bar(st), kc, rowB, pnl);
                        if (leader) ptx::mbar_arrive_expect_tx(full_bar(st), (2u * tx_cta) >> a.tx_shift);
                        else ptx::mbar_arrive_cluster(full_bar(st), 0);
                    }
                }
                if (a.sync_lead > 0 && leader && s.last_in_win)
                    asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(a.win_done + s.win) : "memory");
            }
        }
    } else if (warp == 1 && leader) {
        // ===================================== MMA issuer =======================================
        Sched sc;
        sc.init(a, worker);
        Seg s;
        uint32_t it = 0;
        while (sc.next(s)) {
            if (s.first && !a.resident) {   // resident accumulators are written once per launch: nothing to wait for
                mbar_wait(tempty_bar((uint32_t)s.slot), (uint32_t)(s.use & 1) ^ 1u, a.err, 2);
                ptx::tc_fence_after();
            }
            const uint32_t d_tmem = tmem_base + (uint32_t)s.col;
            const uint32_t idesc = make_instr_desc<CG, KIND>((uint32_t)s.n_eff);
            for (int kb = s.kb0; kb < s.kb1; ++kb, ++it) {
                const uint32_t st = it % C::STAGES, ph = (it / C::STAGES) & 1u;
                mbar_wait(full_bar(st), ph, a.err, 3);
                ptx::tc_fence_after();
                if (issuer) {
                    const uint64_t adesc = make_smem_desc(sA(st));
                    const uint64_t bdesc = make_smem_desc((CG == 2 && (s.flags & kTileSelfB) != 0) ? sA(st) : sB(st));
                    uint32_t acc = (s.first && kb == s.kb0) ? 0u : 1u;
#pragma unroll
                    for (int k = 0; k < kKBytes / 32; ++k) {           // UMMA_K = 32 bytes of K
                        if constexpr (KIND == 3)
                            ptx::umma_ss_mxf4<CG>(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, acc, tmem_base + kSfCol,
                                                  tmem_base + kSfCol + 4);
                        else
                            ptx::umma_ss<CG, KIND>(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, acc);
                        acc = 1u;
                    }
                    ptx::umma_commit<CG>(empty_bar(st));               // frees the smem stage (both CTAs)
                }
                __syncwarp();
            }
            if (s.flush) {
                if (issuer) ptx::umma_commit<CG>(tfull_bar((uint32_t)s.slot));   // accumulator complete -> epilogue
                __syncwarp();
            }
        }
        if (a.prof != nullptr && issuer) a.prof[(size_t)blockIdx.x * 4 + 2] = globaltimer_ns();
    } else if (warp >= 4) {
        // ===================================== epilogue =========================================
        const int q = warp & 3;   // TMEM lane quarter this warp may read
        Sched sc;
        sc.init(a, worker);
        Seg s;
        while (sc.next(s)) {
            if (!s.flush) continue;
            const uint32_t bar_i = (uint32_t)s.slot;
            mbar_wait(tfull_bar(bar_i), (uint32_t)(s.use & 1), a.err, 4);
            ptx::tc_fence_after();
            const bool filler = (CG == 2) && cta_rank != 0 && (s.flags & kTileFiller) != 0;
            const int colbase = ((CG == 2 && cta_rank != 0) ? s.rowA1 : s.rowA0) + q * 32;   // sample of the A row, lane 0
            const int col = colbase + (int)lane;
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)s.col;
            const int row_end = min(a.row_limit, s.rowB + s.n_eff);         // B rows this tile owns
            const int nchunks = filler ? 0 : (s.n_eff + 31) / 32;
#pragma unroll 1
            for (int c = 0; c < nchunks; ++c) {
                const int rbase = s.rowB + c * 32;
                if (rbase >= row_end) break;
                // A chunk wholly above the diagonal is the mirror image of a cell the lower triangle already gets --
                // unless this tile computes a 128-block above the diagonal IN PLACE of its mirror image (exact block
                // cover): then the chunk is written transposed, S[col][row].
                bool xpose = false;
                if (rbase + 31 < colbase) {
                    if ((s.flags & kTileXpose) == 0 || (rbase >> 7) >= (colbase >> 7)) continue;
                    xpose = true;
                }
                uint32_t r[32];
                ptx::tmem_ld_32x32b_x32(taddr + (uint32_t)(c * 32), r);
                ptx::tmem_ld_wait();
                // owner-rows mode: the (at most two) ranks that own rows of this 32-row chunk; a transposed chunk
                // writes row `col`, one owner per lane
                int32_t* own_lo = nullptr;
                int32_t* own_hi = nullptr;
                int own_split = 0;
                if (a.num_peers != 0 && a.peer_mode == 1) {
                    const int probe = xpose ? col : rbase;
                    int o = 0;
                    while (o + 1 < a.num_peers && probe >= a.own_end[o]) ++o;
                    own_split = xpose ? 0x7fffffff : a.own_end[o];
                    own_lo = a.peer[o];
                    own_hi = a.peer[min(o + 1, a.num_peers - 1)];
                }
                // Two cells per atomic: counts are non-negative and every sum stays below 2^31, so a 64-bit add of
                // (cell c | cell c + 1 << 32) never carries between the halves.  Lane pairs trade one value per two
                // rows (the even lane takes row 2 jj of both columns, the odd lane row 2 jj + 1), which halves the
                // number of reds -- the L2 / NVLink atomic rate, not bytes, is what the flush runs against.  Needs an
                // even row pitch (8-byte alignment of an even column); transposed chunks scatter and stay 32-bit.
                if (!xpose && a.red64 != 0 && (a.n_cols & 1) == 0) {
#pragma unroll
                    for (int jj = 0; jj < 16; ++jj) {
                        const int row0 = rbase + 2 * jj, row1 = row0 + 1;
                        int v0, v1;
                        if constexpr (KIND == 0) { v0 = (int)r[2 * jj]; v1 = (int)r[2 * jj + 1]; }
                        else { v0 = __float2int_rn(__uint_as_float(r[2 * jj])); v1 = __float2int_rn(__uint_as_float(r[2 * jj + 1])); }
                        if (!(row0 < row_end && col < a.n_cols && row0 >= col)) v0 = 0;
                        if (!(row1 < row_end && col < a.n_cols && row1 >= col)) v1 = 0;
                        const int got = __shfl_xor_sync(0xffffffffu, (lane & 1) ? v0 : v1, 1);
                        const int srow = (lane & 1) ? row1 : row0;
                        const unsigned long long packed = (lane & 1)
                            ? ((unsigned long long)(unsigned)got | ((unsigned long long)(unsigned)v1 << 32))
                            : ((unsigned long long)(unsigned)v0 | ((unsigned long long)(unsigned)got << 32));
                        if (packed != 0ull) {
                            const size_t o = (size_t)srow * (size_t)a.n_cols + (size_t)(col & ~1);
                            if (a.num_peers == 0) {
                                asm volatile("red.global.add.u64 [%0], %1;" ::"l"(a.S + o), "l"(packed) : "memory");
                            } else if (a.peer_mode == 1) {
                                int32_t* dst = (srow >= own_split ? own_hi : own_lo) + o;
                                asm volatile("red.relaxed.sys.global.add.u64 [%0], %1;" ::"l"(dst), "l"(packed) : "memory");
                            } else {
                                for (int d = 0; d < a.num_peers; ++d)
                                    asm volatile("red.relaxed.sys.global.add.u64 [%0], %1;" ::"l"(a.peer[d] + o), "l"(packed)
                                                 : "memory");
                            }
                        }
                    }
                    continue;
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int row = rbase + j;
                    if (row < row_end && col < a.n_cols && (xpose || row >= col)) {
                        int v;
                        if constexpr (KIND == 0) v = (int)r[j];
                        else v = __float2int_rn(__uint_as_float(r[j]));
                        if (v != 0) {
                            // cell (srow, scol) of S: the lower-triangle position of this product
                            const int srow = xpose ? col : row, scol = xpose ? row : col;
                            const size_t o = (size_t)srow * (size_t)a.n_cols + (size_t)scol;
                            if (a.num_peers == 0) {
                                asm volatile("red.global.add.s32 [%0], %1;" ::"l"(a.S + o), "r"(v) : "memory");
                            } else if (a.peer_mode == 1) {
                                // fused reduce-scatter: one red, into the Gram of the rank that owns this row
                                int32_t* dst = (srow >= own_split ? own_hi : own_lo) + o;
                                asm volatile("red.relaxed.sys.global.add.s32 [%0], %1;" ::"l"(dst), "r"(v) : "memory");
                            } else {
                                // fused reduceByKey: the same red, once per rank, on peer-mapped Gram buffers
                                for (int d = 0; d < a.num_peers; ++d)
                                    asm volatile("red.relaxed.sys.global.add.s32 [%0], %1;" ::"l"(a.peer[d] + o), "r"(v)
                                                 : "memory");
                            }
                        }
                    }
                }
            }
            ptx::tc_fence_before();
            if (!a.resident) {   // hand the accumulator back to the MMA issuer (double buffering of the large-N schedule)
                if constexpr (CG == 1) ptx::mbar_arrive(tempty_bar(bar_i));
                else ptx::mbar_arrive_cluster(tempty_bar(bar_i), 0);
            }
        }
    }

    ptx::tc_fence_before();
    if constexpr (CG == 2) ptx::cluster_sync(); else __syncthreads();
    if (warp == 2) ptx::tmem_dealloc<CG>(tmem_base, kTmemCols);
    if (a.prof != nullptr && threadIdx.x == 0) a.prof[(size_t)blockIdx.x * 4 + 3] = globaltimer_ns();
}

// ---------------------------------------------------------------------------------------------------
// Adaptive stream-K split.  Workers do not all run at the same speed: with int8 operands the kernel needs ~64 B/clk
// per SM from L2 and the SMs of some GPCs get visibly less (measured: per-worker MMA time 1.7 .. 2.4 ms for equal
// shares), so an equal split waits for the slowest pair.  After every sufficiently long launch this kernel turns the
// per-worker timestamps into speeds (units / time) and moves the shares of the next launch towards them.  The Gram
// stays exact whatever the split is (integer atomics); shares are clamped so that a worker never spans more than
// the two tiles it has TMEM accumulators for.
__global__ void rebalance_kernel(const long long* __restrict__ prof, double* __restrict__ cum, int workers, int cta_group,
                                 double gain, double max_share, long long min_ns, int* __restrict__ gen, const TileDesc* __restrict__ tiles,
                                 int num_tiles, int total_weight, int kbw, int col_limit) {
    __shared__ double sh[1024];
    __shared__ double cand[1025];
    __shared__ double red_sum, red_min;
    __shared__ int reject, need_repair;
    const int w = threadIdx.x;
    const bool active = w < workers;
    double t = 0.0, share_old = 0.0;
    if (active) {
        const long long t0 = prof[(size_t)w * cta_group * 4 + 0], t1 = prof[(size_t)w * cta_group * 4 + 2];
        t = (double)(t1 - t0);
        share_old = cum[w + 1] - cum[w];
    }
    sh[w] = active ? t : 1e30;
    if (w == 0) {
        reject = 0;
        need_repair = 0;
    }
    __syncthreads();
    if (w == 0) {
        double mn = 1e30, mx = 0.0;
        for (int i = 0; i < workers; ++i) {
            mn = fmin(mn, sh[i]);
            mx = fmax(mx, sh[i]);
        }
        // too short to time, or already balanced to within 3 %: keep the shares (hysteresis against noise)
        red_min = (mn < (double)min_ns || (mx - mn) < 0.03 * mx) ? -1.0 : mn;
    }
    __syncthreads();
    if (red_min < 0.0) return;
    const double speed = active ? share_old / t : 0.0;
    sh[w] = speed;
    __syncthreads();
    if (w == 0) {
        double sum = 0.0;
        for (int i = 0; i < workers; ++i) sum += sh[i];
        red_sum = sum;
    }
    __syncthreads();
    double share = 0.0;
    if (active) {
        const double est = speed / red_sum;
        share = (1.0 - gain) * share_old + gain * est;
        const double avg = 1.0 / workers;
        share = fmin(fmax(share, 0.5 * avg), max_share * avg);
    }
    __syncthreads();
    sh[w] = share;
    __syncthreads();
    if (w == 0) {
        double sum = 0.0;
        for (int i = 0; i < workers; ++i) sum += sh[i];
        double acc = 0.0;
        cand[0] = 0.0;
        for (int i = 0; i < workers; ++i) {
            acc += sh[i] / sum;
            cand[i + 1] = (i + 1 == workers) ? 1.0 : acc;
        }
    }
    __syncthreads();
    // Repair, then publish: a worker whose pieces under the candidate split would not fit TMEM (more than kMaxSegs
    // accumulators or more than col_limit columns: e.g. the tail of one tile, a whole 13-unit tile and the head of a
    // third) stops at the edge of the tile that does not fit, and its neighbour starts there.  One thread walks the
    // workers in order; the tile cursor only moves forward, so the walk is O(workers + tiles).
    // common case: every worker's pieces fit under the candidate as it is -- checked by all workers in parallel; only
    // when one does not, one thread walks the workers in order and repairs (tens of microseconds: kept off the usual path)
    if (active) {
        const long long uw = (long long)total_weight * kbw;
        const long long ub = (long long)((double)uw * cand[w]);
        const long long ue = (w + 1 == workers) ? uw : (long long)((double)uw * cand[w + 1]);
        int hint = 0;
        if (feasible_end(tiles, num_tiles, ub, ue, kbw, col_limit, hint) < ue) atomicExch(&need_repair, 1);
    }
    __syncthreads();
    if (need_repair && w == 0 && !repair_split(tiles, num_tiles, workers, (long long)total_weight * kbw, kbw, col_limit, cand)) reject = 1;
    __syncthreads();
    if (reject) return;
    if (w <= workers) cum[w] = cand[w];
    if (w == 0) *gen += 1;
}

__global__ void symmetrize_kernel(int32_t* __restrict__ S, int n) {
    // block (bx >= by): read lower tile (bx, by), write it transposed into the upper tile (by, bx)
    __shared__ int32_t tile[32][33];
    const int bx = blockIdx.x, by = blockIdx.y;
    if (bx < by) return;
    const int tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
    for (int r = ty; r < 32; r += 8) {
        const int row = bx * 32 + r, col = by * 32 + tx;
        tile[r][tx] = (row < n && col < n) ? S[(size_t)row * n + col] : 0;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int row = by * 32 + r, col = bx * 32 + tx;   // target (upper)
        if (row < n && col < n && row < col) S[(size_t)row * n + col] = tile[tx][r];
    }
}

__global__ void add_i32_kernel(int32_t* __restrict__ dst, const int32_t* __restrict__ src, int64_t count) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < count; i += stride) dst[i] += src[i];
}

struct PeerPtrs {
    int32_t* p[kMaxPeers];
};

__global__ void add_i32_peers_kernel(PeerPtrs dst, int npeers, const int32_t* __restrict__ src, int64_t count) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < count; i += stride) {
        const int v = src[i];
        if (v != 0)
            for (int d = 0; d < npeers; ++d)
                asm volatile("red.relaxed.sys.global.add.s32 [%0], %1;" ::"l"(dst.p[d] + i), "r"(v) : "memory");
    }
}

struct OwnEnds {
    int e[kMaxPeers];
};

__device__ __forceinline__ int owner_of_row(const OwnEnds& own, int npeers, int row) {
    int q = 0;
    while (q + 1 < npeers && row >= own.e[q]) ++q;
    return q;
}

// Staged partition -> owners: element (row, col) of the lower triangle is added into the Gram of the row's owner.
__global__ void add_i32_owner_kernel(PeerPtrs dst, OwnEnds own, int npeers, const int32_t* __restrict__ src, int n) {
    for (int row = blockIdx.x; row < n; row += gridDim.x) {
        int32_t* d = dst.p[owner_of_row(own, npeers, row)] + (size_t)row * n;
        const int32_t* s = src + (size_t)row * n;
        for (int c = threadIdx.x; c <= row; c += blockDim.x) {
            const int v = s[c];
            if (v != 0) asm volatile("red.relaxed.sys.global.add.s32 [%0], %1;" ::"l"(d + c), "r"(v) : "memory");
        }
    }
}

// All-gather after the reduce-scatter: every rank pulls the lower-triangle part of the rows it does not own from the
// owner's Gram (peer loads over NVLink, 16-byte when the row pitch allows).
__global__ void __launch_bounds__(256) gather_rows_kernel(PeerPtrs src, int32_t* __restrict__ dst, OwnEnds own, int npeers,
                                                          int rank, int n) {
    const bool vec = (n & 3) == 0;
    for (int row = blockIdx.x; row < n; row += gridDim.x) {
        const int q = owner_of_row(own, npeers, row);
        if (q == rank) continue;
        const int32_t* s = src.p[q] + (size_t)row * n;
        int32_t* d = dst + (size_t)row * n;
        if (vec) {
            const int4* s4 = reinterpret_cast<const int4*>(s);
            int4* d4 = reinterpret_cast<int4*>(d);
            for (int c = threadIdx.x; c < (row + 4) / 4; c += blockDim.x) d4[c] = s4[c];   // up to 3 cells past the diagonal: zeros
        } else {
            for (int c = threadIdx.x; c <= row; c += blockDim.x) d[c] = s[c];
        }
    }
}

// The same all-gather as posted writes: every rank pushes the lower-triangle part of the rows it owns into the Gram of
// every other rank (remote stores are fire-and-forget; remote loads pay a NVLink round trip each).
__global__ void __launch_bounds__(256) push_rows_kernel(PeerPtrs dst, const int32_t* __restrict__ src, OwnEnds own,
                                                        int npeers, int rank, int n) {
    const bool vec = (n & 3) == 0;
    const int row_lo = rank == 0 ? 0 : own.e[rank - 1], row_hi = own.e[rank];
    for (int row = row_lo + blockIdx.x; row < row_hi; row += gridDim.x) {
        const int32_t* s = src + (size_t)row * n;
        if (vec) {
            const int4* s4 = reinterpret_cast<const int4*>(s);
            for (int c = threadIdx.x; c < (row + 4) / 4; c += blockDim.x) {
                const int4 v = s4[c];
                for (int d = 0; d < npeers; ++d)
                    if (d != rank) reinterpret_cast<int4*>(dst.p[d] + (size_t)row * n)[c] = v;
            }
        } else {
            for (int c = threadIdx.x; c <= row; c += blockDim.x) {
                const int v = s[c];
                for (int d = 0; d < npeers; ++d)
                    if (d != rank) dst.p[d][(size_t)row * n + c] = v;
            }
        }
    }
}

// All-rank barrier over peer-mapped flag words: rank r publishes `epoch` in slot r of every rank's flag array, then
// waits until every slot of its own array shows it.  One thread per peer.
__global__ void peer_barrier_kernel(PeerPtrs flags, int npeers, int rank, int epoch) {
    const int d = threadIdx.x;
    if (d < npeers) {
        __threadfence_system();
        asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(flags.p[d] + rank), "r"(epoch) : "memory");
        int v;
        const long long t0 = globaltimer_ns();
        do {
            asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(flags.p[rank] + d) : "memory");
            // a peer that died or never reached the barrier must surface as an error, not hang the box
            if (v < epoch && globaltimer_ns() - t0 > 30000000000LL) __trap();
        } while (v < epoch);
    }
    __syncthreads();
    __threadfence_system();
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

template <int CG, int KIND>
cudaError_t launch(const CUtensorMap& tmap, const CUtensorMap& tmap_half, const GramArgs& args, int grid, cudaStream_t stream) {
    using C = Cfg<CG, KIND>;
    // per launch, not cached: the attribute is per device and one process may drive several GPUs
    cudaError_t ea = cudaFuncSetAttribute(gram_kernel<CG, KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    if (ea != cudaSuccess) return ea;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = C::SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, gram_kernel<CG, KIND>, tmap, tmap_half, args);
}

}  // namespace

// Process-wide memory of the speed-weighted splits the rebalancer converged to: the per-worker speeds it measures are a
// property of the device (which SMs get how much L2 bandwidth), so a new context for the same (device, cohort size, tile
// list, window) starts from the split the last one ended with instead of relearning it over its first launches.
namespace {
struct SplitKey {
    int dev, n, rows, tiles, kbw, workers, elem;
    bool operator<(const SplitKey& o) const {
        return std::tie(dev, n, rows, tiles, kbw, workers, elem) <
               std::tie(o.dev, o.n, o.rows, o.tiles, o.kbw, o.workers, o.elem);
    }
};
std::mutex g_split_mu;
std::map<SplitKey, std::vector<double>> g_splits;
}  // namespace

static void remember_split(GramPlan& plan) {
    if (plan.d_cum == nullptr || plan.cum_workers <= 0 || !plan.adaptive) return;
    if (plan.own_hi > plan.own_lo && plan.num_peers <= 1) return;   // a band's tile list is not the cohort's
    std::vector<double> cum((size_t)plan.cum_workers + 1);
    if (cudaMemcpy(cum.data(), plan.d_cum, cum.size() * sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    std::lock_guard<std::mutex> lk(g_split_mu);
    g_splits[SplitKey{plan.cum_dev, plan.cum_for_n, plan.cum_for_rows, plan.cum_tiles, plan.cum_kbw, plan.cum_workers, plan.cum_elem}] = std::move(cum);
}

void gram_plan_free(GramPlan& plan) {
    remember_split(plan);
    if (plan.d_tiles) cudaFree(plan.d_tiles);
    plan.h_tiles.clear();
    if (plan.d_err) cudaFreeHost(plan.d_err);
    if (plan.d_win_done) cudaFree(plan.d_win_done);
    if (plan.d_prof) cudaFree(plan.d_prof);
    if (plan.d_cum) cudaFree(plan.d_cum);
    plan.d_cum = nullptr;
    plan.d_win_done = nullptr;
    plan.d_prof = nullptr;
    plan.d_tiles = nullptr;
    plan.d_err = nullptr;
    plan.tiles_for_n = -1;
}

int gram_read_profile(GramPlan& plan, long long* out, int max_ctas) {
    if (plan.d_prof == nullptr) return 0;
    const int ctas = std::min(max_ctas, std::min(1024, plan.num_sms));
    if (cudaMemcpy(out, plan.d_prof, (size_t)ctas * 4 * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    return ctas;
}

// Tile list of the lower triangle of S.
//   exact == false (kind::mxf4): BM x BN rectangles that touch row >= col, in strips of 8 row blocks walked column by
//     column, so that a run of ~num_sms / 2 consecutive tiles (one wave of the large-N schedule) is a compact patch of S.
//   exact == true: the exact block cover.  Units: 128 x 128 blocks (col block c, row block r), needed iff c <= r.  A tile
//     multiplies `cg` A (column) blocks -- any blocks, one per CTA -- with one or two adjacent B (row) blocks.  With
//     cta_group::2 a tile holds an even number of blocks of every row it touches, but row r needs r + 1 of them, so for
//     r = 4t the block (col 4t, row 4t + 2) is taken out of row 4t + 2 and computed in row 4t as its mirror image
//     (col 4t + 2, row 4t), written transposed: both rows become even and every needed block is covered exactly once.
//     Two-row tiles come first, one-row tiles last (a worker's accumulators must fit the 512 TMEM columns).
static void make_tiles(int n, int cg, bool exact, int bn, int row_lo, int row_hi, bool self_b, std::vector<TileDesc>& out,
                       int* num_full) {
    // [row_lo, row_hi): the rows of S to produce (the whole triangle, or the band an owner-computes context stores)
    out.clear();
    auto n_eff = [&](int row0, int want) { return std::min(want, ((n - row0) + 15) & ~15); };
    if (!exact) {
        // B strips of nearly equal width: ceil(n / 16) units of 16 rows dealt over ceil(n / bn) strips (2504 samples,
        // bn = 240: 3 strips of 240 rows and 8 of 224 instead of 10 of 240 and one of 104).  Tiles of nearly equal
        // weight keep every worker of the resident schedule inside two tiles (two accumulators) under an even split.
        const int BM = 128 * cg;
        const int span = row_hi - row_lo;
        const int nbn = (span + bn - 1) / bn, nbm = (n + BM - 1) / BM;
        const int units = (span + 15) / 16;
        std::vector<int> row0(nbn + 1, row_lo);
        for (int b = 0; b < nbn; ++b) row0[b + 1] = row0[b] + 16 * (units / nbn + (b < units % nbn ? 1 : 0));
        constexpr int kStrip = 8;
        for (int bb = 0; bb < nbn; bb += kStrip)
            for (int am = 0; am < nbm; ++am)
                for (int b = bb; b < std::min(nbn, bb + kStrip); ++b) {
                    const int max_row = std::min(row_hi, row0[b + 1]) - 1;
                    if (am * BM > max_row) continue;   // wholly above the diagonal
                    TileDesc t{};
                    t.rowA0 = am * BM;
                    t.rowA1 = am * BM + 128;
                    t.rowB = row0[b];
                    t.n_eff = std::min(row0[b + 1], ((row_hi + 15) & ~15)) - row0[b];
                    t.acc_cols = bn;
                    // diagonal tile whose 256 B rows are exactly the two A blocks of the pair: CTA r's half of B is its own
                    // A block, so the MMA reads B through the A tile and the producer loads nothing for B (half the
                    // L2 -> SM bytes of the tile)
                    if (self_b && cg == 2 && t.rowB == t.rowA0 && t.n_eff == 2 * 128) t.flags |= kTileSelfB;
                    out.push_back(t);
                }
    } else {
        const int nb = (n + 127) / 128;
        std::vector<TileDesc> two, one;
        auto emit = [&](std::vector<TileDesc>& dst, int c0, int c1, int r0, int rows, bool filler) {
            TileDesc t{};
            t.rowA0 = c0 * 128;
            t.rowA1 = c1 * 128;
            t.rowB = r0 * 128;
            t.n_eff = n_eff(r0 * 128, rows * 128);
            t.acc_cols = (t.n_eff + 31) & ~31;
            t.flags = kTileXpose | (filler ? kTileFiller : 0);
            dst.push_back(t);
        };
        // column blocks each row block needs (a value > the row index = the mirror image of a block of a later row)
        std::vector<std::vector<int>> need(nb);
        for (int r = 0; r < nb; ++r)
            for (int c = 0; c <= r; ++c) need[r].push_back(c);
        if (cg == 2)
            for (int r = 0; r + 2 < nb; r += 4) {
                need[r].push_back(r + 2);                                        // (col r + 2, row r): transposed
                need[r + 2].erase(std::find(need[r + 2].begin(), need[r + 2].end(), r));
            }
        for (int r0 = 0; r0 < nb; r0 += 2) {
            const bool pair = r0 + 1 < nb;
            std::vector<int> common, left0, left1;
            if (pair) {
                for (int c : need[r0])
                    if (std::find(need[r0 + 1].begin(), need[r0 + 1].end(), c) != need[r0 + 1].end()) common.push_back(c);
                if (cg == 2 && (common.size() & 1)) common.pop_back();          // an odd one out joins the one-row tiles
            }
            for (int c : need[r0])
                if (std::find(common.begin(), common.end(), c) == common.end()) left0.push_back(c);
            if (pair)
                for (int c : need[r0 + 1])
                    if (std::find(common.begin(), common.end(), c) == common.end()) left1.push_back(c);
            for (size_t i = 0; i < common.size(); i += cg) emit(two, common[i], common[cg == 2 ? i + 1 : i], r0, 2, false);
            for (int side = 0; side < (pair ? 2 : 1); ++side) {
                const std::vector<int>& left = side == 0 ? left0 : left1;
                for (size_t i = 0; i < left.size(); i += cg) {
                    const bool filler = cg == 2 && i + 1 >= left.size();
                    emit(one, left[i], filler ? left[i] : left[cg == 2 ? i + 1 : i], r0 + side, 1, filler);
                }
            }
        }
        // large-N schedule: whole-tile waves want equal tiles that share row panels of X -- the full-weight two-row
        // tiles go in front, in strips of 8 row blocks walked column pair by column pair (a wave of ~74 consecutive
        // tiles is then a compact patch of S that needs ~34 row blocks of X instead of ~150)
        auto mid = std::stable_partition(two.begin(), two.end(), [&](const TileDesc& t) { return t.n_eff == 256; });
        std::stable_sort(two.begin(), mid, [](const TileDesc& x, const TileDesc& y) {
            const int sx = x.rowB / 1024, sy = y.rowB / 1024;
            if (sx != sy) return sx < sy;
            const int cx = std::min(x.rowA0, x.rowA1) / 256, cy = std::min(y.rowA0, y.rowA1) / 256;
            if (cx != cy) return cx < cy;
            return x.rowB < y.rowB;
        });
        *num_full = (int)(mid - two.begin());
        out = two;
        out.insert(out.end(), one.begin(), one.end());
    }
    if (!exact) *num_full = (int)out.size();   // the rectangles go out in whole-tile waves whatever their edge trim
    int w = 0;
    for (auto& t : out) {
        t.wstart = w;
        w += t.n_eff >> 4;
    }
}

static cudaError_t build_tiles(GramPlan& plan, int n, bool exact, int BN, int row_lo, int row_hi, cudaStream_t stream) {
    std::vector<TileDesc> tiles;
    int num_full = 0;
    make_tiles(n, plan.cta_group, exact, BN, row_lo, row_hi, plan.self_b, tiles, &num_full);
    if (plan.d_tiles) cudaFree(plan.d_tiles);
    plan.d_tiles = nullptr;
    cudaError_t e = cudaMalloc(&plan.d_tiles, tiles.size() * sizeof(TileDesc));
    if (e != cudaSuccess) return e;
    e = cudaMemcpyAsync(plan.d_tiles, tiles.data(), tiles.size() * sizeof(TileDesc), cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) return e;
    e = cudaStreamSynchronize(stream);   // `tiles` is a stack vector
    plan.h_tiles.assign(reinterpret_cast<const int32_t*>(tiles.data()),
                        reinterpret_cast<const int32_t*>(tiles.data() + tiles.size()));
    plan.num_tiles = (int)tiles.size();
    plan.num_full = num_full;
    plan.total_weight = tiles.empty() ? 0 : tiles.back().wstart + (tiles.back().n_eff >> 4);
    plan.tiles_for_n = n;
    plan.tiles_for_cg = plan.cta_group;
    plan.tiles_for_bn = exact ? -1 : BN;
    plan.tiles_row_lo = row_lo;
    plan.tiles_row_hi = row_hi;
    plan.tiles_col_limit = (!exact && BN == kUmmaNScaled) ? (int)kSfCol : (int)kTmemCols;   // mxf4: scale columns at 480
    return e;
}

// Resident schedule (accumulators stay in TMEM for the whole launch) iff the equal split of a window of `kbw` k-blocks,
// after the same repair the rebalancer applies (a worker stops at the edge of a tile whose accumulator would not fit any
// more), lets every worker keep its pieces in the TMEM columns available (those beside the block scales for
// kind::mxf4).  `cum` receives that initial split (workers + 1 fractions).
static bool initial_split(const GramPlan& plan, int workers, int kbw, std::vector<double>& cum) {
    if (plan.total_weight <= 0) return false;
    const TileDesc* tiles = reinterpret_cast<const TileDesc*>(plan.h_tiles.data());
    const long long uw = (long long)plan.total_weight * kbw;
    cum.resize((size_t)workers + 1);
    for (int w = 0; w <= workers; ++w) cum[w] = (double)w / (double)workers;
    if (!repair_split(tiles, plan.num_tiles, workers, uw, kbw, plan.tiles_col_limit, cum.data())) return false;
    for (int w = 0; w < workers; ++w) {   // belt and braces: what the kernel will plan from these fractions must fit
        const long long ub = (long long)((double)uw * cum[w]);
        const long long ue = (w + 1 == workers) ? uw : (long long)((double)uw * cum[w + 1]);
        SegPlan p;
        plan_segments(tiles, plan.num_tiles, 0, ub, ue, kbw, p);
        if (p.overflow || p.cols > plan.tiles_col_limit) return false;
    }
    return true;
}

// Host-only introspection of the schedule (no device needed): the tile list for n samples, and the pieces
// (tile, k-block range, TMEM column) each worker owns in a window of `kbw` k-blocks under an equal split.
int gram_debug_tiles(int n, int cta_group, int exact, int32_t* out, int max_tiles) {
    std::vector<TileDesc> tiles;
    int num_full = 0;
    make_tiles(n, cta_group == 1 ? 1 : 2, exact != 0, exact ? kUmmaN : kUmmaNScaled, 0, n, true, tiles, &num_full);
    const int cnt = std::min<int>((int)tiles.size(), max_tiles);
    if (out != nullptr && cnt > 0) memcpy(out, tiles.data(), (size_t)cnt * sizeof(TileDesc));
    return (int)tiles.size();
}

// Projecting context: A blocks over the n_fit columns of S, B strips over all n_total rows of X (row >= col).  For
// n_total == n_fit this is exactly the tile list of a plain context.
int gram_debug_projection_tiles(int n_fit, int n_total, int cta_group, bool mxf4, int32_t* out, int max_tiles) {
    std::vector<TileDesc> tiles;
    int num_full = 0;
    make_tiles(n_fit, cta_group == 1 ? 1 : 2, false, mxf4 ? kUmmaNScaled : kUmmaN, 0, n_total, true, tiles, &num_full);
    const int cnt = std::min<int>((int)tiles.size(), max_tiles);
    if (out != nullptr && cnt > 0) memcpy(out, tiles.data(), (size_t)cnt * sizeof(TileDesc));
    return (int)tiles.size();
}

int gram_debug_band_tiles(int n, int cta_group, int row_lo, int row_hi, int32_t* out, int max_tiles) {
    std::vector<TileDesc> tiles;
    int num_full = 0;
    make_tiles(n, cta_group == 1 ? 1 : 2, false, kUmmaN, row_lo, row_hi, true, tiles, &num_full);
    const int cnt = std::min<int>((int)tiles.size(), max_tiles);
    if (out != nullptr && cnt > 0) memcpy(out, tiles.data(), (size_t)cnt * sizeof(TileDesc));
    return (int)tiles.size();
}

int gram_debug_plan(const int32_t* tiles8, int num_tiles, int workers, int kbw, int32_t* out, int max_pieces) {
    // the split a first launch uses: equal shares, repaired like initial_split does
    const TileDesc* tiles = reinterpret_cast<const TileDesc*>(tiles8);
    if (num_tiles <= 0) return 0;
    const int col_limit = tiles[0].acc_cols == kUmmaNScaled ? (int)kSfCol : (int)kTmemCols;
    std::vector<double> cum((size_t)workers + 1);
    for (int w = 0; w <= workers; ++w) cum[w] = (double)w / (double)workers;
    return gram_debug_repair(tiles8, num_tiles, workers, kbw, col_limit, cum.data(), out, max_pieces);
}

// Host-only: the rebalancer's repair step on a caller-supplied split (cum: workers + 1 fractions, in / out) followed by
// the plan it yields, in the same format as gram_debug_plan.  -1000: no feasible repair.
int gram_debug_repair(const int32_t* tiles8, int num_tiles, int workers, int kbw, int col_limit, double* cum, int32_t* out,
                      int max_pieces) {
    const TileDesc* tiles = reinterpret_cast<const TileDesc*>(tiles8);
    if (num_tiles <= 0) return 0;
    const long long total = tiles[num_tiles - 1].wstart + (tiles[num_tiles - 1].n_eff >> 4);
    const long long uw = total * kbw;
    if (!repair_split(tiles, num_tiles, workers, uw, kbw, col_limit, cum)) return -1000;
    int cnt = 0;
    for (int w = 0; w < workers; ++w) {
        const long long ub = (long long)((double)uw * cum[w]);
        const long long ue = (w + 1 == workers) ? uw : (long long)((double)uw * cum[w + 1]);
        SegPlan p;
        plan_segments(tiles, num_tiles, 0, ub, ue, kbw, p);
        if (p.overflow || p.cols > col_limit) return -1 - w;
        for (int i = 0; i < p.n; ++i, ++cnt)
            if (cnt < max_pieces) {
                int32_t* o = out + (size_t)cnt * 6;
                o[0] = w; o[1] = p.tile[i]; o[2] = p.lo[i]; o[3] = p.hi[i]; o[4] = p.col[i]; o[5] = p.cols;
            }
    }
    return cnt;
}

cudaError_t gram_accumulate(GramPlan& plan, const void* d_x, int elem_bits, int n, int n_rows, int64_t nv, int64_t ld,
                            int64_t panel, int32_t* d_S, cudaStream_t stream, std::string* err) {
    if (nv <= 0) return cudaSuccess;
    EncodeTiledFn encode = get_encode_fn();
    if (encode == nullptr) {
        if (err) *err = "cuTensorMapEncodeTiled entry point not available";
        return cudaErrorNotSupported;
    }
    if (plan.num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&plan.num_sms, cudaDevAttrMultiProcessorCount, dev);
        const char* cg = getenv("VPCA_CTA_GROUP");
        if (cg != nullptr) plan.cta_group = (atoi(cg) == 1) ? 1 : 2;
        const char* kw = getenv("VPCA_KB_WINDOW");
        if (kw != nullptr) plan.kb_window = atoi(kw);
        const char* sl = getenv("VPCA_SYNC_LEAD");
        if (sl != nullptr) plan.sync_lead = atoi(sl);
        const char* pf = getenv("VPCA_GRAM_PROF");
        plan.profile = (pf != nullptr && atoi(pf) != 0);
        const char* ad = getenv("VPCA_ADAPTIVE");
        if (ad != nullptr) plan.adaptive = atoi(ad) != 0;
        const char* mx = getenv("VPCA_E2M1_MXF4");
        if (mx != nullptr) plan.e2m1_mxf4 = atoi(mx) != 0;
        const char* sb = getenv("VPCA_SELF_B");
        if (sb != nullptr) plan.self_b = atoi(sb) != 0;
        const char* r64 = getenv("VPCA_RED64");
        if (r64 != nullptr) plan.red64 = atoi(r64) != 0;
        const char* gain = getenv("VPCA_REBALANCE_GAIN");
        if (gain != nullptr) plan.gain = std::min(1.0, std::max(0.1, atof(gain)));
        const char* ex = getenv("VPCA_EXACT_COVER");
        if (ex != nullptr) plan.exact_cover = atoi(ex) != 0;
    }
    if (plan.d_win_done == nullptr) {
        cudaError_t e = cudaMalloc(&plan.d_win_done, GramPlan::kMaxWindows * sizeof(int));
        if (e != cudaSuccess) return e;
    }
    if ((plan.profile || plan.adaptive) && plan.d_prof == nullptr) {
        cudaError_t e = cudaMalloc(&plan.d_prof, 1024 * 4 * sizeof(long long));
        if (e != cudaSuccess) return e;
        e = cudaMemsetAsync(plan.d_prof, 0, 1024 * 4 * sizeof(long long), stream);
        if (e != cudaSuccess) return e;
    }
    if (plan.d_err == nullptr) {
        cudaError_t e = cudaHostAlloc(&plan.d_err, 4 * sizeof(int), cudaHostAllocMapped);
        if (e != cudaSuccess) return e;
        for (int i = 0; i < 4; ++i) plan.d_err[i] = 0;
    }
    const bool mxf4 = (elem_bits == 4 && plan.e2m1_mxf4);
    const int tile_bn = mxf4 ? kUmmaNScaled : kUmmaN;
    // Owner-computes band (a context that stores only rows [own_lo, own_hi) of S and has no peers to flush to): only the
    // tiles of those rows are enumerated -- the caller feeds every variant of the cohort to every band's context and no
    // cell is produced twice anywhere (SURVEY 8e "shard output tiles across GPUs ... no reduction").
    const bool banded = plan.own_hi > plan.own_lo && plan.num_peers <= 1;
    const int row_lo = banded ? plan.own_lo : 0, row_hi = banded ? plan.own_hi : n_rows;
    const bool exact = !mxf4 && plan.exact_cover && !banded;   // kind::mxf4 keeps 256 x 240 rectangles (block scales in TMEM)
    if ((banded || exact || plan.num_peers > 1) && n_rows != n) {
        if (err) *err = "projected rows need the rectangle tiling without peers or bands";
        return cudaErrorNotSupported;
    }
    if (plan.tiles_for_n != n || plan.tiles_for_cg != plan.cta_group || plan.tiles_for_bn != (exact ? -1 : tile_bn) ||
        plan.tiles_row_lo != row_lo || plan.tiles_row_hi != row_hi) {
        cudaError_t e = build_tiles(plan, n, exact, tile_bn, row_lo, row_hi, stream);
        if (e != cudaSuccess) return e;
    }
    if (panel > 0) {
        if ((panel % 128) != 0) {
            if (err) *err = "panel_variants must be a multiple of 128";
            return cudaErrorInvalidValue;
        }
        ld = panel;   // rows of a panel are `panel` cells apart, panels n * panel cells apart
    }
    const uintptr_t align = (elem_bits == 4) ? 31 : 15;
    if ((reinterpret_cast<uintptr_t>(d_x) & align) != 0 || (((ld * elem_bits) / 8) & align) != 0 ||
        (elem_bits == 4 && (ld % 128) != 0)) {
        if (err) *err = "dense tile must be 16-byte aligned with a 16-byte multiple row pitch (32 / ld % 128 == 0 for e2m1)";
        return cudaErrorInvalidValue;
    }

    const int cgp = plan.cta_group;
    const int workers = (cgp == 2) ? plan.num_sms / 2 : plan.num_sms;
    // one k-block = one 128-byte swizzle atom of shared memory: 128 int8, 64 bf16 or 128 e2m1 cells (TMA expands
    // 4-bit cells to one byte each, CU_TENSOR_MAP_DATA_TYPE_16U4_ALIGN16B)
    const int elems_per_kb = (elem_bits == 16) ? 64 : (mxf4 ? 256 : 128);
    const int kind = (elem_bits == 8) ? 0 : (elem_bits == 16 ? 1 : (mxf4 ? 3 : 2));
    if (mxf4 && panel > 0 && (panel % 256) != 0) {
        if (err) *err = "kind::mxf4 needs panel_variants % 256 == 0";
        return cudaErrorInvalidValue;
    }

    CUtensorMap tmap;
    // Panel layout: dim0 = cells of one panel row, dim1 = samples, dim2 = panels.  Row-major input is one panel as
    // wide as the tile.  e2m1: globalDim[0] must be a multiple of 128 (the caller guarantees zero cells up to there).
    const int64_t npanels = panel > 0 ? (nv + panel - 1) / panel : 1;
    const int64_t dim0 = panel > 0 ? panel : (elem_bits == 4 ? (mxf4 ? ((nv + 1) / 2) * 2 : ((nv + 127) / 128) * 128) : nv);
    // rows of X: all n_rows samples (fitted, then projected); S has n columns
    const cuuint64_t gdim[3] = {(cuuint64_t)dim0, (cuuint64_t)n_rows, (cuuint64_t)npanels};
    const cuuint64_t gstride[2] = {(cuuint64_t)ld * (cuuint64_t)elem_bits / 8,
                                   (cuuint64_t)n_rows * (cuuint64_t)ld * (cuuint64_t)elem_bits / 8};
    const cuuint32_t box[3] = {(cuuint32_t)elems_per_kb, (cuuint32_t)kBoxRows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUtensorMapDataType tmtype = elem_bits == 8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8
                                       : (elem_bits == 16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                                          : (mxf4 ? CU_TENSOR_MAP_DATA_TYPE_16U4_ALIGN8B
                                                                  : CU_TENSOR_MAP_DATA_TYPE_16U4_ALIGN16B));
    CUresult r = encode(&tmap, tmtype, 3,
                        const_cast<void*>(d_x), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        if (err) *err = "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r);
        return cudaErrorInvalidValue;
    }
    // the same tensor with a 64-row box: the B operand of the N <= 128 tiles of the exact block cover (cta_group::2)
    CUtensorMap tmap_half;
    const cuuint32_t box_half[3] = {(cuuint32_t)elems_per_kb, (cuuint32_t)(kBoxRows / 2), 1};
    r = encode(&tmap_half, tmtype, 3, const_cast<void*>(d_x), gdim, gstride, box_half, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        if (err) *err = "cuTensorMapEncodeTiled (64-row box) failed with CUresult " + std::to_string((int)r);
        return cudaErrorInvalidValue;
    }

    GramArgs args{};
    // a band is addressed through the virtual origin of the full matrix: row r lives at d_S + (r - own_lo) * n
    args.S = banded ? d_S - (ptrdiff_t)plan.own_lo * n : d_S;
    args.num_peers = (plan.num_peers > 1 && d_S == plan.peer_base[plan.peer_rank]) ? plan.num_peers : 0;
    for (int d = 0; d < kMaxPeers; ++d) args.peer[d] = d < plan.num_peers ? plan.peer_S[d] : nullptr;
    args.peer_mode = plan.peer_mode;
    for (int d = 0; d < kMaxPeers; ++d) args.own_end[d] = plan.own_end[d];
    args.tiles = static_cast<const TileDesc*>(plan.d_tiles);
    cudaHostGetDevicePointer(reinterpret_cast<void**>(&args.err), plan.d_err, 0);
    args.n_cols = n;
    args.num_tiles = plan.num_tiles;
    args.num_full = plan.num_full;
    args.total_weight = plan.total_weight;
    args.kb_total = (int)((nv + elems_per_kb - 1) / elems_per_kb);
    args.kb_per_panel = panel > 0 ? (int)(panel / elems_per_kb) : args.kb_total;
    args.num_workers = workers;
    args.elems_per_kb = elems_per_kb;
    args.acc_stride = mxf4 ? kUmmaNScaled : kUmmaN;
    args.col_limit = plan.tiles_col_limit;
    args.row_limit = row_hi;
    args.red64 = plan.red64 ? 1 : 0;
    {
        int kbw = plan.kb_window;
        if (kbw <= 0 && panel > 0) kbw = args.kb_per_panel;   // one L2 window per panel
        if (kbw <= 0) {
            // window of X sized to ~32 MiB so that every tile re-reads it from L2 (126 MB) rather than HBM
            const long long target = 32ll << 20;
            kbw = (int)std::max<long long>(8, std::min<long long>(4096, target / ((long long)n_rows * kKBytes)));
        }
        kbw = std::min(kbw, args.kb_total);
        // cheap upper bound first (a worker with less than a tile's worth of work can touch few tiles), then the exact test
        std::vector<double> cum0;
        args.resident = (plan.num_tiles <= 4 * workers && initial_split(plan, workers, kbw, cum0)) ? 1 : 0;
        int dev = 0;
        cudaGetDevice(&dev);
        args.kb_window = args.resident ? kbw : args.kb_total;
        // the device-side split (speed-weighted by rebalance_kernel from launch to launch) starts from the repaired
        // equal split; it is only meaningful for one (workers, tile list, window length)
        if (args.resident && (plan.d_cum == nullptr || plan.cum_workers != workers || plan.cum_tiles != plan.num_tiles ||
                              plan.cum_kbw != kbw || plan.cum_for_n != n || plan.cum_for_rows != n_rows ||
                              plan.cum_elem != elem_bits)) {
            remember_split(plan);
            if (plan.adaptive && !banded) {   // a split learned earlier on this device for the same schedule, if it still fits TMEM
                std::lock_guard<std::mutex> lk(g_split_mu);
                auto it = g_splits.find(SplitKey{dev, n, n_rows, plan.num_tiles, kbw, workers, elem_bits});
                if (it != g_splits.end()) {
                    std::vector<double> learned = it->second;
                    const TileDesc* tiles = reinterpret_cast<const TileDesc*>(plan.h_tiles.data());
                    if (repair_split(tiles, plan.num_tiles, workers, (long long)plan.total_weight * kbw, kbw, plan.tiles_col_limit,
                                     learned.data()))
                        cum0 = learned;
                }
            }
            if (plan.d_cum) cudaFree(plan.d_cum);
            plan.d_cum = nullptr;
            cudaError_t e = cudaMalloc(&plan.d_cum, (size_t)(workers + 2) * sizeof(double) + sizeof(int));
            if (e != cudaSuccess) return e;
            cum0.push_back(0.0);                                   // [workers + 1]: unused
            cum0.push_back(0.0);                                   // [workers + 2]: the update counter (int)
            e = cudaMemcpyAsync(plan.d_cum, cum0.data(), (size_t)(workers + 2) * sizeof(double) + sizeof(int),
                                cudaMemcpyHostToDevice, stream);   // pageable source: staged before the call returns
            if (e != cudaSuccess) return e;
            plan.cum_workers = workers;
            plan.cum_tiles = plan.num_tiles;
            plan.cum_kbw = kbw;
            plan.cum_for_n = n;
            plan.cum_for_rows = n_rows;
            plan.cum_dev = dev;
            plan.cum_elem = elem_bits;
        }
    }
    plan.last_resident = args.resident;
    const int nwin = (args.kb_total + args.kb_window - 1) / args.kb_window;
    const long long uw = (long long)args.total_weight * args.kb_window;
    args.active_workers = (int)std::min<long long>(workers, uw);
    args.sync_lead = (args.resident && nwin <= GramPlan::kMaxWindows) ? plan.sync_lead : 0;
    args.win_done = plan.d_win_done;
    const bool adapt = plan.adaptive && args.resident && workers <= 1024 && args.active_workers == workers;
    args.prof = (plan.profile || adapt) ? plan.d_prof : nullptr;
    args.cum = plan.d_cum;
    args.tx_shift = (elem_bits == 4 && !mxf4 && getenv("VPCA_E2M1_TX_FULL") == nullptr) ? 1 : 0;
    if (args.sync_lead > 0) {
        cudaError_t e = cudaMemsetAsync(plan.d_win_done, 0, (size_t)nwin * sizeof(int), stream);
        if (e != cudaSuccess) return e;
    }

    const int grid = workers * cgp;
    cudaError_t le;
    if (cgp == 2)
        le = kind == 0 ? launch<2, 0>(tmap, tmap_half, args, grid, stream)
                       : (kind == 1 ? launch<2, 1>(tmap, tmap_half, args, grid, stream)
                                    : (kind == 2 ? launch<2, 2>(tmap, tmap_half, args, grid, stream) : launch<2, 3>(tmap, tmap_half, args, grid, stream)));
    else
        le = kind == 0 ? launch<1, 0>(tmap, tmap_half, args, grid, stream)
                       : (kind == 1 ? launch<1, 1>(tmap, tmap_half, args, grid, stream)
                                    : (kind == 2 ? launch<1, 2>(tmap, tmap_half, args, grid, stream) : launch<1, 3>(tmap, tmap_half, args, grid, stream)));
    if (le != cudaSuccess) return le;
    if (adapt) {
        // shares move towards the measured speeds, at most 35 % above the mean; a split under which some worker's
        // accumulators would not fit TMEM is rejected by the kernel itself
        rebalance_kernel<<<1, 1024, 0, stream>>>(plan.d_prof, plan.d_cum, workers, cgp, plan.gain, 1.35, 300000,
                                                 reinterpret_cast<int*>(plan.d_cum + workers + 2), static_cast<const TileDesc*>(plan.d_tiles), plan.num_tiles,
                                                 plan.total_weight, args.kb_window, plan.tiles_col_limit);
        le = cudaGetLastError();
    }
    return le;
}

// Loads every kernel of this translation unit on the current device.  With CUDA's lazy module loading the FIRST launch of
// a kernel loads it, and that load can wait for the device to go idle; a host thread that has just enqueued a spinning
// peer_barrier_kernel for one context and then launches a not-yet-loaded kernel (for this or another context of the same
// process) would wait for a barrier that can only complete once the thread has enqueued the other contexts' barriers --
// a deadlock (observed on B200 with two contexts in one process: the 30 s barrier watchdog fired).  One process driving
// several contexts (vpca_gram_set_peers_local, vpca_pool) therefore loads everything up front: cudaFuncGetAttributes
// for all kernels, plus an empty launch of those that are enqueued behind a barrier.
cudaError_t gram_preload_kernels(cudaStream_t stream) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaSuccess;
#define VPCA_LOAD(k) if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, k)
    VPCA_LOAD((gram_kernel<1, 0>)); VPCA_LOAD((gram_kernel<1, 1>)); VPCA_LOAD((gram_kernel<1, 2>)); VPCA_LOAD((gram_kernel<1, 3>));
    VPCA_LOAD((gram_kernel<2, 0>)); VPCA_LOAD((gram_kernel<2, 1>)); VPCA_LOAD((gram_kernel<2, 2>)); VPCA_LOAD((gram_kernel<2, 3>));
    VPCA_LOAD(rebalance_kernel); VPCA_LOAD(symmetrize_kernel); VPCA_LOAD(add_i32_kernel); VPCA_LOAD(add_i32_peers_kernel);
    VPCA_LOAD(add_i32_owner_kernel); VPCA_LOAD(gather_rows_kernel); VPCA_LOAD(push_rows_kernel); VPCA_LOAD(peer_barrier_kernel);
#undef VPCA_LOAD
    if (e != cudaSuccess) return e;
    PeerPtrs pp{};
    OwnEnds own{};
    peer_barrier_kernel<<<1, 32, 0, stream>>>(pp, 0, 0, 0);                 // npeers = 0: no thread touches a flag
    push_rows_kernel<<<1, 32, 0, stream>>>(pp, nullptr, own, 0, 0, 0);        // own.e[0] = 0: no rows
    gather_rows_kernel<<<1, 32, 0, stream>>>(pp, nullptr, own, 0, 0, 0);      // n = 0
    add_i32_owner_kernel<<<1, 32, 0, stream>>>(pp, own, 0, nullptr, 0);       // n = 0
    add_i32_peers_kernel<<<1, 32, 0, stream>>>(pp, 0, nullptr, 0);            // count = 0
    add_i32_kernel<<<1, 32, 0, stream>>>(nullptr, nullptr, 0);
    symmetrize_kernel<<<dim3(1, 1), dim3(32, 8), 0, stream>>>(nullptr, 0);    // n = 0: every access is masked
    return cudaGetLastError();
}

// How many clusters of `cluster_size` CTAs of the int8 Gram kernel (1 CTA per SM: ~200 KB of shared memory each) the
// current device can hold at once -- the GPC layout decides whether a 4- or 8-CTA cluster (TMA multicast of a shared
// operand) could still use every SM.  Diagnostic only.
int gram_debug_max_clusters(int cluster_size) {
    using C = Cfg<2, 0>;
    if (cudaFuncSetAttribute(gram_kernel<2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES) != cudaSuccess) return -1;
    if (cluster_size > 8 &&
        cudaFuncSetAttribute(gram_kernel<2, 0>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) return -1;
    int sms = 0, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(sms / cluster_size * cluster_size));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = C::SMEM_BYTES;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cluster_size;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int clusters = 0;
    if (cudaOccupancyMaxActiveClusters(&clusters, gram_kernel<2, 0>, &cfg) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    return clusters;
}

cudaError_t gram_symmetrize(int32_t* d_S, int n, cudaStream_t stream) {
    const int nb = (n + 31) / 32;
    symmetrize_kernel<<<dim3(nb, nb), dim3(32, 8), 0, stream>>>(d_S, n);
    return cudaGetLastError();
}

cudaError_t gram_add(int32_t* d_dst, const int32_t* d_src, int64_t count, cudaStream_t stream) {
    add_i32_kernel<<<592, 256, 0, stream>>>(d_dst, d_src, count);
    return cudaGetLastError();
}

cudaError_t gram_add_peers(GramPlan& plan, const int32_t* d_src, int64_t count, cudaStream_t stream) {
    PeerPtrs pp{};
    for (int d = 0; d < plan.num_peers; ++d) pp.p[d] = plan.peer_S[d];
    add_i32_peers_kernel<<<592, 256, 0, stream>>>(pp, plan.num_peers, d_src, count);
    return cudaGetLastError();
}

cudaError_t gram_add_owners(GramPlan& plan, const int32_t* d_src, int n, cudaStream_t stream) {
    PeerPtrs pp{};
    OwnEnds own{};
    for (int d = 0; d < plan.num_peers; ++d) pp.p[d] = plan.peer_S[d];
    for (int d = 0; d < kMaxPeers; ++d) own.e[d] = plan.own_end[d];
    add_i32_owner_kernel<<<592, 256, 0, stream>>>(pp, own, plan.num_peers, d_src, n);
    return cudaGetLastError();
}

cudaError_t gram_gather_rows(GramPlan& plan, int32_t* d_S, int n, cudaStream_t stream) {
    PeerPtrs pp{};
    OwnEnds own{};
    for (int d = 0; d < plan.num_peers; ++d) pp.p[d] = plan.peer_S[d];
    for (int d = 0; d < kMaxPeers; ++d) own.e[d] = plan.own_end[d];
    // VPCA_GATHER=push (default) | pull | copy: posted peer stores, peer loads, or copy-engine 2-D copies per band
    const char* how = getenv("VPCA_GATHER");
    if (how != nullptr && strcmp(how, "pull") == 0) {
        gather_rows_kernel<<<1184, 256, 0, stream>>>(pp, d_S, own, plan.num_peers, plan.peer_rank, n);
    } else if (how != nullptr && strcmp(how, "copy") == 0) {
        for (int q = 0; q < plan.num_peers; ++q) {
            if (q == plan.peer_rank) continue;
            const int r0 = q == 0 ? 0 : plan.own_end[q - 1], r1 = plan.own_end[q];
            cudaError_t e = cudaMemcpy2DAsync(d_S + (size_t)r0 * n, (size_t)n * 4, plan.peer_S[q] + (size_t)r0 * n,
                                              (size_t)n * 4, (size_t)std::min(n, r1) * 4, (size_t)(r1 - r0),
                                              cudaMemcpyDeviceToDevice, stream);
            if (e != cudaSuccess) return e;
        }
    } else {
        push_rows_kernel<<<1184, 256, 0, stream>>>(pp, d_S, own, plan.num_peers, plan.peer_rank, n);
    }
    return cudaGetLastError();
}

cudaError_t gram_peer_barrier(GramPlan& plan, cudaStream_t stream) {
    PeerPtrs pp{};
    for (int d = 0; d < plan.num_peers; ++d) pp.p[d] = plan.peer_flags[d];
    plan.peer_epoch += 1;
    peer_barrier_kernel<<<1, 32, 0, stream>>>(pp, plan.num_peers, plan.peer_rank, plan.peer_epoch);
    return cudaGetLastError();
}

}  // namespace vpca

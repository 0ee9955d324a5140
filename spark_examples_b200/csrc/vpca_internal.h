// Internal declarations shared by the libvpca translation units (not part of the ABI).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <string>
#include <vector>

#include "../../include/vpca.h"

namespace vpca {

// ---- Gram (gram_sm100.cu) --------------------------------------------------------------------
struct GramPlan {
    int cta_group = 2;        // tcgen05 cta_group (1: 128x256 tiles per CTA, 2: 256x256 per CTA pair)
    int kb_window = 0;        // k-blocks per L2 window (0 -> automatic)
    int num_sms = 0;
    void* d_tiles = nullptr;  // device tile list (TileDesc, gram_sm100.cu)
    std::vector<int32_t> h_tiles;   // the same list on the host (8 ints per tile): resident / TMEM-fit decisions
    int num_tiles = 0;
    int num_full = 0;         // leading full-weight tiles (whole-tile waves of the large-N schedule)
    int total_weight = 0;     // sum over tiles of n_eff / 16
    int tiles_col_limit = 512;   // TMEM columns the accumulators of one worker may take
    bool exact_cover = false; // VPCA_EXACT_COVER=1: the exact 128-block cover of the lower triangle (4.5 % fewer MMAs at
                              // 2504 samples) instead of square 256 x 256 tiles.  Off by default: its N = 128 tiles need
                              // 96 B/clk per SM from L2 (A 16 KB + B 8 KB per 256 MMA cycles) where the 256 x 256 tiles
                              // need 64, and L2 -> SM bandwidth is what the kernel runs against -- measured on B200:
                              // 2.06 ms vs 1.65 ms per 2504 x 1M Gram (profiles/README.md, round 2)
    int tiles_for_n = -1;     // n_samples the tile list was built for
    int tiles_for_cg = 0;
    int tiles_for_bn = 0;
    int tiles_row_lo = 0, tiles_row_hi = 0;   // rows of S the tile list covers
    int own_lo = 0, own_hi = 0;   // band-only context: the rows of S it stores (own_hi == 0: the whole matrix); without
                                  // peers the Gram kernel then computes exactly those rows (owner-computes)
    bool e2m1_mxf4 = true;    // packed e2m1 cells run through kind::mxf4 (2x MMA rate, unit block scales);
                              // VPCA_E2M1_MXF4=0 selects kind::f8f6f4 (TMA-expanded cells, int8 rate)
    int last_resident = 0;
    int* d_err = nullptr;     // device debug words written before a watchdog trap
    static constexpr int kMaxWindows = 1 << 16;
    int sync_lead = 0;        // VPCA_SYNC_LEAD: windows a worker may lead the slowest one by (0 = no pacing; measured
                              // on B200: pacing only slows every worker to the slowest one, see DESIGN.md)
    int* d_win_done = nullptr;
    bool self_b = true;       // VPCA_SELF_B=0: diagonal tiles load their B rows although they are the pair's own A blocks
    bool red64 = true;        // VPCA_RED64=0: one 32-bit red per cell in the flush instead of two cells per 64-bit red
    double gain = 0.5;        // VPCA_REBALANCE_GAIN: how far a launch moves the shares towards the measured speeds (measured on
                              // B200, 2504 x 1M int8: 0.5 settles at 1.61 ms within three launches, 0.7 and 1.0 hover at 1.70)
    bool adaptive = true;     // VPCA_ADAPTIVE=0 keeps the stream-K split equal instead of speed-weighted
    double* d_cum = nullptr;  // cumulative worker shares (workers + 1 doubles) + update counter
    int cum_workers = 0, cum_tiles = 0, cum_kbw = 0, cum_for_n = 0, cum_for_rows = 0, cum_dev = 0, cum_elem = 0;   // what the
                                                                                    // split in d_cum was made for
    // fused multi-GPU reduction: Gram buffers / barrier flags of all ranks, peer-mapped through CUDA IPC
    int num_peers = 0, peer_rank = 0, peer_epoch = 0;
    int32_t* peer_S[16] = {};     // Gram of rank d as seen from this device: the address of row 0 (for a rank that stores
                                  // only a row band this is a VIRTUAL origin, valid for the rows of the band only)
    int32_t* peer_base[16] = {};  // start of rank d's allocation (what an IPC mapping must be closed with)
    int32_t* peer_flags[16] = {};
    int band_row0[16] = {}, band_rows[16] = {};   // rows rank d stores (band_rows 0 or n: all of them)
    bool peers_ipc = false;       // peer mappings came from cudaIpcOpenMemHandle (other processes), not from peer access
    int peer_mode = 0;        // 0: every flush goes to all ranks' Grams; 1: to the owner of the row only (+ gather)
    int own_end[16] = {};     // peer_mode 1: rank q owns Gram rows [own_end[q-1], own_end[q])
    bool profile = false;     // VPCA_GRAM_PROF=1: per-CTA timestamps in d_prof
    long long* d_prof = nullptr;
};
// Copies the per-CTA timestamps of the last profiled launch (4 per CTA) to host; returns the CTA count.
int gram_read_profile(GramPlan& plan, long long* out, int max_ctas);

// S(lower triangle, row >= col) += X X^T for the nv variants of a dense sample-major tile.
//   d_x : device, element (s, v) at index s * ld + v; elem_bits 8 (int8), 16 (bf16) or 4 (packed e2m1: two cells per
//         byte, ld % 128 == 0 and zero cells up to the next multiple of 128 variants)
//   d_S : device int32 n_rows x n row-major (pitch n): rows [0, n) the fitted Gram, rows [n, n_rows) the cross block of
//         the projected samples (n_rows == n: a plain context).  Only cells with row >= col < n are written.
// Returns cudaSuccess or the first CUDA error; never synchronises.
// panel > 0: the tile is stored as ceil(nv / panel) consecutive panels of `panel` variants, each panel n rows of
// `panel` cells (cell (s, v) at (v / panel) * n * panel + s * panel + v % panel, zero cells after nv in the last
// panel); `ld` is ignored.  Keeps the pages touched per L2 window few (a row-major tile with a multi-MB pitch puts
// every sample row on its own 2 MB page and thrashes the TLBs).
cudaError_t gram_accumulate(GramPlan& plan, const void* d_x, int elem_bits, int n, int n_rows, int64_t nv, int64_t ld,
                            int64_t panel, int32_t* d_S, cudaStream_t stream, std::string* err);
cudaError_t gram_symmetrize(int32_t* d_S, int n, cudaStream_t stream);
cudaError_t gram_add(int32_t* d_dst, const int32_t* d_src, int64_t count, cudaStream_t stream);
cudaError_t gram_add_peers(GramPlan& plan, const int32_t* d_src, int64_t count, cudaStream_t stream);
cudaError_t gram_add_owners(GramPlan& plan, const int32_t* d_src, int n, cudaStream_t stream);
cudaError_t gram_gather_rows(GramPlan& plan, int32_t* d_S, int n, cudaStream_t stream);
cudaError_t gram_peer_barrier(GramPlan& plan, cudaStream_t stream);
cudaError_t gram_preload_kernels(cudaStream_t stream);   // see gram_sm100.cu: lazy module loading vs spinning barriers
cudaError_t encode_preload_kernels();
void gram_plan_free(GramPlan& plan);
int gram_debug_max_clusters(int cluster_size);
int gram_debug_band_tiles(int n, int cta_group, int row_lo, int row_hi, int32_t* out, int max_tiles);
int gram_debug_projection_tiles(int n_fit, int n_total, int cta_group, bool mxf4, int32_t* out, int max_tiles);
int gram_debug_tiles(int n, int cta_group, int exact, int32_t* out, int max_tiles);
int gram_debug_plan(const int32_t* tiles8, int num_tiles, int workers, int kbw, int32_t* out, int max_pieces);
int gram_debug_repair(const int32_t* tiles8, int num_tiles, int workers, int kbw, int col_limit, double* cum, int32_t* out,
                      int max_pieces);

// ---- encode (encode.cu) ------------------------------------------------------------------------
// CSR rows [0, nv) (d_off has nv+1 entries; entry e of row v is d_idx[d_off[v] - base + ...]) -> dense
// sample-major tile of n rows, zero-filled first.  d_flags[0] is OR-ed with 1 on an index outside [0, n) and 2 on a
// multiplicity overflow.  d_rows (n entries, may be nullptr = identity): the tile row of input sample s.
cudaError_t encode_calls(const int64_t* d_off, int64_t base, const void* d_idx, int idx_bytes, int64_t nv, int n,
                         int elem_bits, int max_mult, void* d_x, int64_t ld, int64_t panel, const int32_t* d_rows,
                         int* d_flags, cudaStream_t stream);   // idx_bytes: 4 (int32) or 2 (uint16)

// Packed rows (`stride` bytes apart) -> dense cells (binary carriers).  code 0: one N-bit bitmap per variant, LSB
// first; code 1 / 2: PLINK .bed rows (2 bits per sample), carriers of A1 / of A2.
cudaError_t encode_bits(const uint8_t* d_bits, int64_t stride, int64_t nv, int n, int elem_bits, void* d_x, int64_t ld,
                        int64_t panel, int code, const int32_t* d_rows, cudaStream_t stream);

// ---- multi-dataset keying: variant keys, join, merge (join.cu) ---------------------------------------------
struct JoinWork {
    uint64_t* d_hash = nullptr;      // 2 per row: MurmurHash3_x64_128 of the variant key
    int32_t* d_table = nullptr;      // open-addressing table of row indices (-1 = empty)
    uint64_t table_slots = 0;
    int64_t* d_rows = nullptr;       // output rows / calls each input row is responsible for, and their exclusive scans
    int64_t* d_len = nullptr;
    int64_t* d_row_base = nullptr;
    int64_t* d_nnz_base = nullptr;
    int32_t* d_leader = nullptr;
    int64_t* d_prefix = nullptr;
    int64_t* d_block = nullptr;      // scan scratch
    int64_t* d_totals = nullptr;     // {output rows, output calls}
    int64_t* h_totals = nullptr;     // pinned copy
    int64_t cap_rows = 0;
    int64_t* d_out_off = nullptr;    // the joined CSR: out_rows + 1 offsets, out_nnz sample indices
    int32_t* d_out_idx = nullptr;
    int64_t cap_out_rows = 0, cap_out_nnz = 0;
    int64_t out_rows = -1, out_nnz = 0;   // result of the last join (-1: none)
    // device copies of the caller's input (grow-only)
    uint8_t* d_payload = nullptr;
    int64_t* d_key_off = nullptr;
    int64_t* d_off = nullptr;
    int32_t* d_idx = nullptr;
    int64_t cap_payload = 0, cap_in_rows = 0, cap_in_nnz = 0;
};
cudaError_t hash_keys(const uint8_t* d_payload, const int64_t* d_off, int64_t nkeys, uint64_t* d_hash, cudaStream_t stream);
cudaError_t join_rows(JoinWork& w, int mode, int variant_set_count, int64_t n_left, const uint8_t* d_payload,
                      const int64_t* d_key_off, const int64_t* d_off, const int32_t* d_idx, int64_t nrows, cudaStream_t stream,
                      int64_t* out_rows, int64_t* out_nnz, int64_t* launches);
void join_free(JoinWork& w);

// ---- centering + eigensolve (eig.cu) ---------------------------------------------------------------
struct EigWork {
    int n = 0;
    double* d_C = nullptr;     // n x n centered matrix, overwritten by the tridiagonalisation
    double* d_rowsum = nullptr;
    double* d_v = nullptr;     // Householder vector of the current step (n)
    double* d_w = nullptr;     // w vector of the current step (n)
    double* d_p = nullptr;     // p = tau A v (n)
    double* d_diag = nullptr;  // n
    double* d_off = nullptr;   // n
    double* d_tau = nullptr;   // n
    double* d_scal = nullptr;  // small scalar scratch
    double* d_mm = nullptr;    // matrixMean of the last center_gram (d_scal[0] does not survive the solvers)
    double* d_evals = nullptr; // k
    double* d_evecs = nullptr; // n x k (column-major)
    double* d_lu = nullptr;    // 8 n scratch for inverse iteration
    int* d_nz = nullptr;
    int* d_step = nullptr;               // {next step, step of the pending trailing update}
    cudaGraphExec_t graph_exec = nullptr; // kGraphSteps tridiagonalisation steps, replayed n / kGraphSteps times
    int graph_n = 0;
    bool graph_fused = false;
    int kmax = 0;
    // Lanczos workspace (allocated on the first Lanczos solve)
    double* d_V = nullptr;      // n x kLzCap orthonormal basis, column-major
    double* d_lzw = nullptr;    // 2 n: w ping-pong
    double* d_lzs = nullptr;    // alpha | beta | h | h2 | e2 | Y | theta2 | res | scal2 | part
    int* d_lzst = nullptr;      // {step, flag, ticket, step cap}
    unsigned* d_lzbar = nullptr;   // grid barrier counter of the persistent Lanczos kernel
    double* d_lzG = nullptr;       // kLzCap x kLzCap: V^T V of the Lanczos basis (one-reduction Gram-Schmidt)
    long long* d_lzprof = nullptr; // VPCA_LZ_PROF=1: phase timestamps of block 0 (first 64 steps)
    bool c_valid = false;       // d_C holds the centred matrix of the last center_gram()
    int lz_blocks = 0;          // blocks of the persistent kernel (= SMs; 0: cooperative launch unavailable or VPCA_LZ_PERSIST=0)
    const int32_t* d_S = nullptr;   // the (symmetrised) int32 Gram the last center_gram() read
    cudaGraphExec_t lz_graph = nullptr;   // kLzChunk Lanczos steps
    int last_method = 0;        // 1 direct, 2 Lanczos, 3 Lanczos abandoned -> direct
    int last_iters = 0;         // Lanczos steps of the last solve
    int mode = 0;               // 0 auto, 1 direct, 2 Lanczos whenever n allows
};
cudaError_t eig_alloc(EigWork& w, int n, int kmax);
void eig_free(EigWork& w);
// row sums + matrix mean always; the FP64 matrix C only when `materialise` (or later, on demand, through center_matrix)
cudaError_t center_gram(EigWork& w, const int32_t* d_S, cudaStream_t stream, bool materialise);
cudaError_t center_matrix(EigWork& w, cudaStream_t stream);
cudaError_t eig_topk(EigWork& w, int k, cudaStream_t stream, int64_t* launches);
// Projection of m cross rows d_X (m x w.n int32, pitch w.n) onto the first k vectors of the last eig_topk, with the row
// sums and matrixMean of the last center_gram: d_y (m x k, column-major).  Scratch: d_rowmean (m), d_part
// (proj_chunks(w.n) * m * k).  Three launches.
int proj_chunks(int n);
cudaError_t eig_project(const EigWork& w, const int32_t* d_X, int m, int k, double* d_rowmean, double* d_part, double* d_y,
                        cudaStream_t stream);

// ---- saved model: loadings and scoring (model.cu) --------------------------------------------------------------
// Every kernel reads an encoded chunk in panel layout: ceil(nv / panel) panels of `rows` x panel cells, zero after nv.
// Loadings of the nv variants of a chunk from its rows [0, n_fit) and the first k columns of U (n_fit x k, column-major,
// EigWork::d_evecs): d_L (nv x k row-major) and d_carriers (nv).  Fixed order over f: bit-identical for any chunking.
cudaError_t model_loadings(const void* d_x, int elem_bits, int64_t nv, int64_t panel, int rows, int n_fit, const double* d_u,
                           int k, double* d_L, int32_t* d_carriers, cudaStream_t stream);
// Scoring of a chunk of m study samples (rows = m): d_acc (m x k doubles, then m int64) += (T, r) of the chunk, where
// variant v uses model row d_mrows[v] of d_L (V x k) / d_n (-1: skipped).  d_scratch: model_score_scratch(m, k) bytes.
size_t model_score_scratch(int m, int k);
cudaError_t model_score(const void* d_x, int elem_bits, int64_t nv, int64_t panel, int m, const int32_t* d_mrows,
                        const double* d_L, const int32_t* d_n, int k, double* d_scratch, double* d_acc, cudaStream_t stream);
// a_c = sum_f u_fc and b_c = sum_f (rs_f / n) u_fc for c < k, fixed order.
cudaError_t model_terms(const double* d_u, const double* d_rowsum, int n, int k, double* d_a, double* d_b, cudaStream_t stream);
// d_dst += d_src, both accumulators of m samples and k columns (doubles, then int64).
cudaError_t model_add(double* d_dst, const double* d_src, int m, int k, cudaStream_t stream);
// d_y (m x kout, column-major) from an accumulator of k columns and d_terms = {lambda[k], a[k], b[k], matrix mean}.
cudaError_t model_finish(const double* d_acc, int m, int k, int kout, int n_fit, const double* d_terms, double* d_y,
                         cudaStream_t stream);

// ---- synthetic generator (synth.cu) ----------------------------------------------------------------
cudaError_t synth_dense(uint64_t seed, int n, int64_t v0, int64_t nv, int mode, int elem_bits, void* d_x,
                        int64_t ld, int64_t panel, cudaStream_t stream);

}  // namespace vpca

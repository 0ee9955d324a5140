/*
 * vpca.h -- C ABI of libvpca.so: the B200-native VariantsPca hot path
 *           (genotype encode -> N x N similarity/Gram accumulation -> centering + top-k eigenvectors).
 *
 * Drop-in boundary.  The reference (googlegenomics/spark-examples) has no FFI; the boundary is the
 * public method set of `class VariantsPcaDriver` as used by `main`
 * (src/main/scala/com/google/cloud/genomics/spark/examples/VariantsPca.scala:38-50).  Each entry
 * point below names the reference lines whose work it replaces; INTEGRATION.md shows the JNI class
 * (`NativePca`) and the Scala changes a maintainer would add to bind them.
 *
 * Conventions
 *   - plain C, no C++/torch types; every pointer is either HOST memory owned by the caller or a raw
 *     CUDA device pointer where the parameter name starts with `d_`.
 *   - every function returns VPCA_OK (0) or a negative vpca_status; vpca_last_error() gives the text.
 *     No C++ exception crosses the ABI.
 *   - a vpca_ctx owns one GPU's worth of state (device buffers, streams, staging); a vpca_pool owns one ctx per GPU
 *     of the box and is what one driver JVM holds (the reference's process model, VariantsPca.scala:38-50).
 *   - threading: accumulate_* / commit / abort may be called concurrently from many threads (the task threads of
 *     `mapPartitions`, VariantsPca.scala:184-189).  Host-input calls run on one of `staging_lanes` private lanes
 *     (streams + staging buffers): the context mutex is held for bookkeeping only, never across a copy, a kernel or
 *     a synchronisation, so the H2D copy and encode of one task overlap the Gram kernel of another.  One partition
 *     id belongs to one thread at a time (spark.speculation off).  reset / finalize / get_* / compute_pca are
 *     driver-side calls made when no accumulate call is in flight.
 *   - device-resident input (on_device tiles, panels) and everything driver-side is ordered on the stream given in
 *     vpca_config.stream (or a private stream); functions that return host data synchronise before returning.
 *   - there is no CPU fallback: vpca_create fails with VPCA_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef VPCA_H_
#define VPCA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VPCA_VERSION_MAJOR 0
#define VPCA_VERSION_MINOR 2

typedef enum vpca_status {
    VPCA_OK = 0,
    VPCA_ERR_BAD_ARG = -1,
    VPCA_ERR_INDEX_OUT_OF_RANGE = -2, /* sample index outside [0, n_samples): the reference would throw
                                         (VariantsPca.scala:59 NoSuchElementException / :188 Breeze bounds) */
    VPCA_ERR_CUDA = -3,
    VPCA_ERR_NCCL = -4,     /* the cross-GPU reduction (`reduceByKey`, VariantsPca.scala:190) cannot run: no peer path
                               between two devices, or a peer mapping failed */
    VPCA_ERR_OVERFLOW = -5, /* an int32 similarity count (VariantsPca.scala:185) could exceed 2^31-1,
                               or a multiplicity does not fit the encoding */
    VPCA_ERR_STATE = -6,
    VPCA_ERR_NOMEM = -7,
    VPCA_ERR_UNSUPPORTED = -8
} vpca_status;

typedef enum vpca_dtype {
    VPCA_DTYPE_I8 = 0,  /* int8 genotype encoding, tcgen05 kind::i8, exact int32 accumulation   */
    VPCA_DTYPE_BF16 = 1, /* bf16 genotype encoding, tcgen05 kind::f16, fp32 TMEM accumulation flushed
                            into the int32 Gram before 2^24 could be reached (exact)              */
    VPCA_DTYPE_E2M1 = 2  /* 4-bit e2m1 cells (0, 1, 2 exact), two per byte in HBM and in shared memory;
                            tcgen05 kind::mxf4 (block-scaled FP4 MMA, unit UE8M0 scales kept in TMEM:
                            twice the int8 MMA rate) with fp32 accumulation, flushed like bf16 (exact).
                            Half the HBM/L2 bytes per cell.  Dense tiles need ld % 128 == 0 (panels:
                            % 256), 32-byte alignment and zero cells up to the next multiple of 128
                            variants; max_multiplicity <= 2.  VPCA_E2M1_MXF4=0 selects kind::f8f6f4
                            (cells expanded to bytes by TMA, int8 rate) instead.                     */
} vpca_dtype;

typedef struct vpca_ctx vpca_ctx;

typedef struct vpca_config {
    uint32_t struct_size;      /* sizeof(vpca_config), for forward compatibility                     */
    int32_t n_samples;         /* N = common.indexes.size (VariantsPca.scala:183,199)                 */
    int32_t device;            /* CUDA device ordinal                                                  */
    int32_t dtype;             /* vpca_dtype                                                           */
    int32_t num_pc;            /* PcaConf.numPc (GenomicsConf.scala:85); default 2 when 0             */
    int32_t max_multiplicity;  /* largest value a genotype cell may take (1 = binary carriers, the
                                  reference rule VariantsPca.scala:58; 2 = dosage / a sample listed
                                  twice).  0 -> 2.  Used for the overflow guards.                     */
    int32_t partitions_in_flight; /* staging Grams for uncommitted partitions; 0 -> 4                 */
    int32_t staging_lanes;     /* host-input calls that may run concurrently on this GPU (each lane: two
                                  streams + double-buffered staging, ~1 GB); 0 -> 2, at most 16            */
    int64_t chunk_variants;    /* variants per device staging chunk for CSR input; 0 -> automatic     */
    int64_t chunk_nnz;         /* sample-index entries per device staging chunk; 0 -> automatic       */
    void* stream;              /* cudaStream_t to order all work on; NULL -> private stream           */
    void* d_gram;              /* optional caller-owned device buffer of n_samples^2 int32 (e.g. the
                                  tensor the host all-reduces with NCCL); NULL -> library-owned       */
    int32_t gram_band_row0;    /* gram_band_rows > 0: this context stores ONLY rows [row0, row0 + rows) of the   */
    int32_t gram_band_rows;    /* Gram -- the band it owns in VPCA_PEER_OWNER_ROWS mode (vpca_owner_row_bands);
                                  for cohorts whose full Gram should not be replicated per GPU (100 k
                                  samples: 40 GB; the reference's sizing note at VariantsPca.scala:176-177).
                                  0 -> the whole matrix                                                 */
} vpca_config;

/* ---- lifecycle ---------------------------------------------------------------------------- */
int vpca_version(void);                                  /* major * 1000 + minor */
int vpca_create(const vpca_config* cfg, vpca_ctx** out); /* replaces `new VariantsPcaDriver(conf)` state
                                                            that lives on the executor side
                                                            (VariantsPca.scala:81-85, :185)             */
int vpca_destroy(vpca_ctx* ctx);
/* Last error text of `ctx` (or of the calling thread when ctx == NULL).  Never NULL. */
const char* vpca_last_error(const vpca_ctx* ctx);
/* Zero the Gram and forget all partitions: start a new analysis on the same ctx. */
int vpca_reset(vpca_ctx* ctx);
/* Wait for everything enqueued on the context's stream (kernels of device-resident input, commits, gathers). */
int vpca_synchronize(vpca_ctx* ctx);
/* Pinned (page-locked, portable) host memory for callers that stage rows themselves -- the JNI binding wraps it in
 * direct ByteBuffers so that Spark tasks pack RDD[Seq[Int]] rows (VariantsPca.scala:153-168) straight into memory the
 * copy engines read at full PCIe rate, with no JVM array pinning. */
int vpca_host_alloc(size_t bytes, void** out);
int vpca_host_free(void* p);

/* ---- encode (VariantsPca.scala:56-60 extractCallInfo, :153-168 getCallsRdd) ---------------------
 * Host-side records arrive already projected to `RDD[Seq[Int]]` rows (CSR: row v = the sample indices
 * with hasVariation at variant v, duplicates allowed, any order; offsets has nv+1 entries).
 * vpca_encode_calls runs ONLY the device encode (CSR -> dense sample-major tile) and copies the tile
 * back: out[s * ld + v] = multiplicity of sample s in row v.  It exists so the encode kernel can be
 * parity-checked on its own; accumulate_calls below fuses it with the Gram.
 * Element type of `out` follows cfg.dtype (int8_t or bf16 bits as uint16_t); ld in elements, >= nv. */
int vpca_encode_calls(vpca_ctx* ctx, const int64_t* offsets, const int32_t* sample_idx, int64_t nv, void* out,
                      int64_t ld);

/* ---- similarity / Gram accumulation (VariantsPca.scala:182-191 getSimilarityMatrix) --------------
 * vpca_accumulate_calls = the body of `mapPartitions` (:184-189) for one batch of rows of Spark
 * partition `partition_id`: encode on device + S_partition += X X^T on tcgen05 tensor cores.  May be
 * called many times per partition.  Nothing is visible in the Gram until vpca_commit(partition_id)
 * (task success); vpca_abort discards it (task failure / retry), so a retried task is counted exactly
 * once -- the property the reference gets from returning a fresh matrix per task (:185).
 * partition_id < 0 means "no staging": accumulate straight into the Gram (single-shot callers). */
int vpca_accumulate_calls(vpca_ctx* ctx, int64_t partition_id, const int64_t* offsets, const int32_t* sample_idx,
                          int64_t nv);
/* Same, with 16-bit sample indices -- halves the host->device bytes of the dominant e2e cost.  Valid whenever
 * n_samples <= 65536, which covers every cohort the reference itself can process (MLlib's RowMatrix refuses more
 * than 65535 columns at VariantsPca.scala:226). */
int vpca_accumulate_calls_u16(vpca_ctx* ctx, int64_t partition_id, const int64_t* offsets, const uint16_t* sample_idx,
                              int64_t nv);
/* Packed wire format (SURVEY 8f-1): one bitmap per variant instead of an index list -- bit s (least significant bit
 * first) of row v is `hasVariation` of sample s (VariantsPca.scala:58), rows stride_bytes apart
 * (>= ceil(n_samples / 8)).  N/8 bytes per variant on the wire whatever the carrier count (313 B at N = 2504 against
 * ~4.3 KB of int32 indices for the synthetic cohort); expanded to cells on the device by a bit-matrix transpose.
 * Binary carriers only (a sample cannot be listed twice).  Same staging / commit semantics as vpca_accumulate_calls. */
int vpca_accumulate_bits(vpca_ctx* ctx, int64_t partition_id, const uint8_t* bits, int64_t nv, int64_t stride_bytes);
/* PLINK 1 .bed rows as they are on disk (variant-major; 2 bits per sample, low bits first: 00 homozygous A1,
 * 01 missing, 10 heterozygous, 11 homozygous A2), rows stride_bytes apart (>= ceil(n_samples / 4)).  `hasVariation`
 * (:58) = "carries the counted allele": counted_allele 1 -> codes {00, 10} (A1, PLINK's minor / alternate allele),
 * 2 -> codes {10, 11}; a missing call carries nothing, like a no-call.  Stands in for the retired ingestion
 * (rdd/VariantsRDD.scala:187-236) at N/4 bytes per variant.  Same staging / commit semantics as vpca_accumulate_calls. */
int vpca_accumulate_bed(vpca_ctx* ctx, int64_t partition_id, const uint8_t* rows, int64_t nv, int64_t stride_bytes,
                        int32_t counted_allele);
int vpca_commit(vpca_ctx* ctx, int64_t partition_id);
int vpca_abort(vpca_ctx* ctx, int64_t partition_id);

/* Pre-encoded dense input, sample-major: x[s * ld + v], s in [0, n_samples), v in [0, nv); element
 * type per cfg.dtype; ld (elements) must make rows 16-byte aligned.  on_device != 0: `x` is a device
 * pointer and is consumed in place (no copy) -- the resident-in-HBM path of bench.py; otherwise it is
 * host memory and is staged through the device in chunks.  Accumulates straight into the Gram. */
int vpca_accumulate_dense(vpca_ctx* ctx, const void* x, int64_t nv, int64_t ld, int on_device);

/* Device-resident input in PANEL layout -- the layout to keep a whole cohort in HBM: the nv variants are cut into
 * panels of `panel_variants` (a multiple of 128); panel p is a contiguous n_samples x panel_variants row-major block,
 * panels follow each other:  cell (s, v) at  (v / P) * n_samples * P + s * P + v % P  (cells; e2m1: two per byte),
 * cells after nv in the last panel are zero, d_x 32-byte aligned.  One Gram launch consumes everything.  Why: with a
 * row-major tile whose rows are megabytes apart every sample row sits on its own 2 MB page and each 128-row TMA box
 * touches 128 pages; panels keep the pages live per L2 window to a few dozen (measured 2x on 2504 x 5M int8). */
int vpca_accumulate_panels(vpca_ctx* ctx, const void* d_x, int64_t nv, int64_t panel_variants);

/* `reduceByKey(_ + _)` (:190) across GPUs is ONE all-reduce of the raw Gram buffer, driven by the host
 * (torch.distributed / NCCL in this repo, see INTEGRATION.md): all-reduce the n_samples^2 int32 at
 * vpca_gram_device_ptr() between the last commit and vpca_finalize_gram().  Until finalize only the
 * lower triangle (row >= col) of the buffer is meaningful. */
int vpca_gram_device_ptr(vpca_ctx* ctx, void** d_gram);
/* Fused alternative to the host-driven all-reduce (one process per GPU, all GPUs of one NVLink box): once every
 * rank has exchanged the 64-byte handle of vpca_gram_export_ipc() and called vpca_gram_set_peers() with the handles
 * of all ranks (rank order; needs a library-owned Gram, vpca_config.d_gram == NULL), the epilogue of the Gram
 * kernel adds every flushed accumulator straight into the Gram of EVERY rank (red.global.add.s32 on peer-mapped
 * memory), so compute and reduceByKey (:190) are one kernel.  Protocol per pass, on every rank:
 *   vpca_reset -> vpca_peer_barrier -> accumulate ... (commit) -> vpca_peer_barrier -> vpca_finalize_gram.
 * vpca_peer_barrier enqueues an all-rank barrier over peer-mapped flags on the context's stream. */
int vpca_gram_export_ipc(vpca_ctx* ctx, void* handle64);
int vpca_gram_set_peers(vpca_ctx* ctx, const void* handles, int32_t world, int32_t rank);
/* The same wiring when ONE process owns all `world` contexts (the reference's process model: one driver JVM whose task
 * threads share the executors' state, VariantsPca.scala:38-50, :184-190): peer access is enabled between the devices and
 * ctxs[r] becomes rank r.  Contexts may share a device (a 1-GPU box exercises the same kernels).  VPCA_ERR_NCCL when two
 * of the devices have no peer path.  vpca_pool_create does this for the contexts it creates. */
int vpca_gram_set_peers_local(vpca_ctx* const* ctxs, int32_t world);
int vpca_peer_barrier(vpca_ctx* ctx);
/* How the fused epilogue reduces across the peers set above:
 *   VPCA_PEER_REPLICATE (default): every flush goes into the Gram of every rank -- world x the remote traffic, no
 *     second phase.  Best at 2 GPUs.
 *   VPCA_PEER_OWNER_ROWS: reduce-scatter + all-gather.  Rank q owns a band of Gram rows (equal shares of the lower
 *     triangle, boundaries on multiples of 32); a flush goes only to the owner of its row, and vpca_gram_gather()
 *     (barrier, pull the rows owned by the other ranks over NVLink, barrier) completes every rank's copy.
 *     Protocol per pass:  vpca_reset -> vpca_peer_barrier -> accumulate ... (commit) -> vpca_gram_gather ->
 *     vpca_finalize_gram.  vpca_gram_gather() is valid in both modes (REPLICATE: just the closing barrier). */
enum { VPCA_PEER_REPLICATE = 0, VPCA_PEER_OWNER_ROWS = 1 };
int vpca_gram_set_peer_mode(vpca_ctx* ctx, int32_t mode);
int vpca_gram_gather(vpca_ctx* ctx);
/* Row bands of VPCA_PEER_OWNER_ROWS: rank q owns Gram rows [row_end[q-1], row_end[q]) (row_end[-1] = 0).  A context
 * created with vpca_config.gram_band_row0 / gram_band_rows set to its band stores nothing else: its kernels still
 * compute the whole lower triangle of their variant shard, but every flush leaves for the owner of its row, the bands
 * ARE the result (no gather), and vpca_get_gram_band reads them.  This is the biobank-scale form (100 k samples: a
 * 40 GB matrix, 2.6 - 14 GB per GPU at 8 GPUs) of `reduceByKey` (VariantsPca.scala:190). */
int vpca_owner_row_bands(int32_t n_samples, int32_t world, int32_t* row_end /* world entries */);
/* Rows [row0, row0 + rows) of the Gram as this context holds them (lower triangle meaningful before finalize;
 * n_samples int32 per row). */
int vpca_get_gram_band(vpca_ctx* ctx, int32_t row0, int32_t rows, int32_t* out);

/* Mirror the lower triangle into the upper one: after this the buffer equals the reference's
 * similarity matrix with all N^2 entries present (:189-190). */
int vpca_finalize_gram(vpca_ctx* ctx);
/* Copy the finalized Gram to host, row-major n_samples x n_samples int32 (the collected
 * RDD[((Int, Int), Int)] in key order). */
int vpca_get_gram(vpca_ctx* ctx, int32_t* out);
/* Checkpoint / resume of a long accumulation (SURVEY 8f-2): copy out / restore the Gram as accumulated so far
 * (committed partitions only, NOT finalized: lower triangle meaningful).  After vpca_load_partial_gram accumulation
 * continues on top of the restored counts; the caller keeps the watermark (which partitions are in it). */
int vpca_get_partial_gram(vpca_ctx* ctx, int32_t* out, int64_t* variants_in_gram /* may be NULL */);
/* variants_in_gram: how many variants the restored counts stand for (what vpca_get_partial_gram reported); they keep
 * counting against the int32 bound of a similarity count (VariantsPca.scala:185). */
int vpca_load_partial_gram(vpca_ctx* ctx, const int32_t* gram, int64_t variants_in_gram);
/* Variants folded into the Gram so far (committed partitions + direct input); negative vpca_status on error. */
int64_t vpca_variant_count(vpca_ctx* ctx);
/* Load a Gram (checkpoint restore / tests); marks it finalized. */
int vpca_set_gram(vpca_ctx* ctx, const int32_t* gram);

/* ---- computePca (VariantsPca.scala:198-231) --------------------------------------------------------
 * Centering (:199-223) in FP64 with the reference's operation order, then the top-k eigenvectors of the
 * centered matrix (= the first k columns of U that MLlib's RowMatrix.computePrincipalComponents returns
 * at :226) by Householder tridiagonalisation + Sturm bisection + inverse iteration on the GPU.
 *   vecs : n_samples x k, column-major -- the layout of `pca.toArray` (:227); vecs[i + c*n] is PC c of
 *          sample i.  Each column is unit-norm and sign-normalised (largest-|.| entry positive).
 *   evals: k eigenvalues of the centered matrix, descending (may be NULL).
 *   non_zero_rows: `rowSums.filter(_ > 0).size` (:207), may be NULL. */
int vpca_compute_pca(vpca_ctx* ctx, int32_t k, double* vecs, double* evals, int32_t* non_zero_rows);
/* The centered matrix itself (row-major N x N doubles) for parity tests of :199-223. */
int vpca_get_centered(vpca_ctx* ctx, double* out);
/* Tridiagonal form of the centered matrix after the last vpca_compute_pca (diag: n, offdiag: n-1). */
int vpca_get_tridiagonal(vpca_ctx* ctx, double* diag, double* offdiag);

/* ---- projection of held-out samples onto the fitted PCs -----------------------------------------------------------
 * The reference fits every callset it reads (VariantsPca.scala:182-231).  A projecting context keeps N FITTED samples
 * (cfg->n_samples; their Gram, centring and PCs are exactly what a plain N-sample context computes) and M PROJECTED ones
 * that are only placed on those axes.  Rows of the context: fitted 0..N-1, projected N..N+M-1.
 *   Cross counts  X_pf = #{variants where projected p and fitted f both carry variation}: the pair loop
 *                 `for (c1 <- callset; c2 <- callset)` (:186-188) restricted to c1 projected, c2 fitted; exact int32 with the
 *                 overflow bound of the Gram (:185).  Stored with the Gram in ONE (N+M) x N row-major buffer: rows 0..N-1
 *                 the fitted Gram (the layout of a plain context), rows N..N+M-1 the cross block; the projected x projected
 *                 counts are neither stored nor computed.  A caller-owned cfg->d_gram must hold (N+M) N int32.
 *   Coordinates   the centring of :199-223 applied to a new row with the FITTED row sums and matrixMean, in the operation
 *                 order of the fitted centring:  rs_p = sum_f X_pf (exact), rowMean_p = rs_p / N,
 *                 c_pf = ((X_pf - rowMean_p) - rowSums_f / N) + matrixMean,   y_pc = (sum_f c_pf u_fc) / lambda_c
 *                 (Gower's add-a-point formula).  The reference has no projection step: these numbers are not pinned by
 *                 it.  Projected coordinates shrink towards 0 relative to fitted ones; no correction is applied.
 * Input: every host-input and join route takes samples in SOURCE order and applies sample_rows on the device.  Pre-encoded
 * input (vpca_accumulate_dense, vpca_accumulate_panels, the synthetic generator) has N+M rows already in row order.
 * Existing entry points on a projecting context: get_gram / compute_pca / get_centered work on the fitted N x N block;
 * get_partial_gram / load_partial_gram copy all (N+M) N counts; set_gram is VPCA_ERR_UNSUPPORTED, and so are
 * vpca_gram_export_ipc / vpca_gram_set_peers / vpca_gram_set_peers_local (multi-GPU runs all-reduce the buffer of
 * vpca_gram_device_ptr), gram_band_rows and VPCA_EXACT_COVER=1 (when M > 0).  The pool does not create projecting contexts. */
typedef struct vpca_projection {
    uint32_t struct_size;          /* sizeof(vpca_projection)                                                              */
    int32_t n_projected;           /* M >= 0; M = 0 gives exactly the context vpca_create makes                           */
    const int32_t* sample_rows;    /* N + M entries: input sample position s -> row of the context (fitted rows 0..N-1,
                                      projected rows N..N+M-1); a permutation of 0..N+M-1, else VPCA_ERR_BAD_ARG.
                                      NULL = identity (the last M inputs are projected).  Copied by the call.              */
} vpca_projection;
int vpca_create_projecting(const vpca_config* cfg, const vpca_projection* proj, vpca_ctx** out);
/* The cross block X (M x N row-major int32) after vpca_finalize_gram: the rows of `matrix(c1, c2)` (:186-190) for c1
 * projected.  M = 0: nothing is written. */
int vpca_get_cross_gram(vpca_ctx* ctx, int32_t* out);
/* Coordinates of the projected samples on the first k PCs of the last vpca_compute_pca (:224-227 extended to new rows):
 * out[p + c * M] = y_pc, M x k column-major (the layout of vecs).  k <= the k of that call, else VPCA_ERR_BAD_ARG; before
 * any vpca_compute_pca since the Gram last changed: VPCA_ERR_STATE.  Fixed reduction order: repeated calls are
 * bit-identical. */
int vpca_project_pca(vpca_ctx* ctx, int32_t k, double* out);
/* ---- saved model: project later without the panel genotypes ------------------------------------------------------
 * Expanding X_pf = sum_v x_pv x_fv in the coordinate of vpca_project_pca gives the same number from per-variant
 * quantities of the fitted panel (u_fc, lambda_c: the PCs of the last vpca_compute_pca; rs_f: the fitted row sums, :206):
 *   loadings  L_vc = sum_f x_fv u_fc (FP64)   carriers  n_v = sum_f x_fv (exact)
 *   col_sums  a_c = sum_f u_fc (~0)            rowsum_dots  b_c = sum_f (rs_f / N) u_fc
 *   T_pc = sum_v x_pv L_vc,  r_p = sum_v x_pv n_v (= rs_p, exact),  y_pc = (((T_pc - (r_p / N) a_c) - b_c) + mean a_c) / lambda_c
 * so {L, n, lambda, a, b, matrixMean} scores any cohort in one pass over its genotypes: no panel genotypes, no Gram and no
 * eigensolve.  Not in the reference (it has no projection step, VariantsPca.scala:224-231): these numbers are not pinned
 * by it.
 *
 * Fit side: a plain or projecting context after vpca_compute_pca; k <= the k of that call (else VPCA_ERR_BAD_ARG; before
 * any vpca_compute_pca since the Gram last changed: VPCA_ERR_STATE).  The loadings calls take the same input as the
 * accumulate calls (a second pass over the same rows), read the fitted rows 0..N-1 only, run on a lane like them and never
 * touch the Gram or the partition staging.  Host outputs, one row per input variant in input order: loadings nv x k
 * row-major, carriers nv.  The reduction over f has a fixed order that depends on f only, so a variant's loadings are
 * bit-identical whatever route, chunking or call delivered it. */
int vpca_pca_loadings_calls(vpca_ctx* ctx, int32_t k, const int64_t* offsets, const int32_t* sample_idx, int64_t nv,
                            double* loadings, int32_t* carriers);
int vpca_pca_loadings_bed(vpca_ctx* ctx, int32_t k, const uint8_t* rows, int64_t nv, int64_t stride_bytes,
                          int32_t counted_allele, double* loadings, int32_t* carriers);
int vpca_pca_loadings_panels(vpca_ctx* ctx, int32_t k, const void* d_x, int64_t nv, int64_t panel_variants,
                             double* loadings, int32_t* carriers);
/* The k eigenvalues, a (col_sums), b (rowsum_dots) and matrixMean of the last vpca_compute_pca (host outputs). */
int vpca_pca_model_terms(vpca_ctx* ctx, int32_t k, double* eigenvalues, double* col_sums, double* rowsum_dots,
                         double* matrix_mean);

/* Scoring side.  A scoring context is a vpca_ctx whose cfg->n_samples are the M study samples; the model is copied to the
 * device by the call.  cfg->d_gram and gram_band_rows must be unset: it allocates no Gram, and its Gram entry points
 * (accumulate_*, finalize, get_gram / get_partial_gram / load_partial_gram / set_gram, compute_pca, project_pca, the
 * peers) return VPCA_ERR_UNSUPPORTED.
 *   vpca_score_calls / _bed: the input of vpca_accumulate_calls / _bed for the study samples, plus model_rows (nv): the
 *     model row of each variant, -1 = not in the model (skipped); a row outside [-1, n_variants) gives
 *     VPCA_ERR_INDEX_OUT_OF_RANGE.  partition_id >= 0: the scores stay private to the partition until vpca_commit (a
 *     partition committed again replaces its earlier scores); vpca_abort discards them.  partition_id < 0: direct input.
 *   vpca_score_panels: device-resident study cells in the panel layout of vpca_accumulate_panels (direct input).
 *   vpca_score_project: out[p + c * M] = y_pc for c < k <= model->k (M x k column-major, like vpca_project_pca); the sum
 *     runs over direct input first (in call order), then the committed partitions in ascending partition id, so the result
 *     depends on how the input was cut into partitions and calls, never on thread timing or commit order.
 *     *matched_variants (may be NULL): input variants with a model row.  VPCA_ERR_STATE while a partition is uncommitted. */
typedef struct vpca_model {
    uint32_t struct_size;          /* sizeof(vpca_model)                                                   */
    int32_t n_fitted, k;           /* N of the fitted panel, columns of the model                          */
    int64_t n_variants;            /* V (< 2^31)                                                           */
    const double* loadings;        /* V x k row-major                                                      */
    const int32_t* carriers;       /* V                                                                    */
    const double* eigenvalues, *col_sums, *rowsum_dots;   /* k each                                    */
    double matrix_mean;
} vpca_model;
int vpca_create_scoring(const vpca_config* cfg, const vpca_model* model, vpca_ctx** out);
int vpca_score_calls(vpca_ctx* ctx, int64_t partition_id, const int64_t* offsets, const int32_t* sample_idx, int64_t nv,
                     const int32_t* model_rows);
int vpca_score_bed(vpca_ctx* ctx, int64_t partition_id, const uint8_t* rows, int64_t nv, int64_t stride_bytes,
                   int32_t counted_allele, const int32_t* model_rows);
int vpca_score_panels(vpca_ctx* ctx, const void* d_x, int64_t nv, int64_t panel_variants, const int32_t* model_rows);
int vpca_score_project(vpca_ctx* ctx, int32_t k, double* out, int64_t* matched_variants /* may be NULL */);

/* Host-only: the tiles (records of vpca_debug_tiles) of a projecting context with n_fit fitted and n_total - n_fit
 * projected samples -- A blocks over the n_fit columns of S, B rows over all n_total rows (row >= col); mxf4 != 0: the
 * 240-wide strips of kind::mxf4, else the 256-wide ones of int8 / bf16.  Returns the tile count (may exceed max_tiles). */
int vpca_debug_projection_tiles(int32_t n_fit, int32_t n_total, int32_t cta_group, int32_t mxf4, int32_t* out,
                                int32_t max_tiles);

/* ---- one process, all GPUs of the box (SURVEY 8b "process model") --------------------------------------------------
 * A vpca_pool is what `class VariantsPcaDriver` holds on a multi-GPU host: one vpca_ctx per GPU, wired with
 * vpca_gram_set_peers_local in VPCA_PEER_OWNER_ROWS mode (VPCA_PEER_REPLICATE when n_samples < 64 x n_gpus).  Spark
 * partition p is served by GPU p % n_gpus (`mapPartitionsWithIndex`, VariantsPca.scala:184); all entry points below
 * except create / destroy / reset / reduce / get / compute may be called concurrently from the task threads.
 *   vpca_pool_create(cfg, n_gpus, devices, &pool)      cfg.device / stream / d_gram / gram_band_* are ignored
 *   task p:  vpca_pool_accumulate_* (pool, p, ...) ...  vpca_pool_commit(pool, p)   |  vpca_pool_abort(pool, p)
 *   driver:  vpca_pool_reduce_and_finalize(pool)        `reduceByKey(_ + _)` (:190): every commit has already been
 *                                                       added into the owners of its Gram rows over NVLink; this is the
 *                                                       closing barrier + all-gather of the bands + symmetrize
 *            vpca_pool_get_gram / vpca_pool_compute_pca  (:189-190, :198-227), served by GPU 0 of the pool */
typedef struct vpca_pool vpca_pool;
int vpca_pool_create(const vpca_config* cfg, int32_t n_gpus, const int32_t* devices /* NULL: 0 .. n_gpus-1 */,
                     vpca_pool** out);
int vpca_pool_destroy(vpca_pool* pool);
int32_t vpca_pool_size(const vpca_pool* pool);
/* The context that serves partition_id (partition_id < 0: GPU 0). */
vpca_ctx* vpca_pool_ctx(vpca_pool* pool, int64_t partition_id);
const char* vpca_pool_last_error(const vpca_pool* pool);
int vpca_pool_reset(vpca_pool* pool);
int vpca_pool_accumulate_calls(vpca_pool* pool, int64_t partition_id, const int64_t* offsets, const int32_t* sample_idx,
                               int64_t nv);
int vpca_pool_accumulate_calls_u16(vpca_pool* pool, int64_t partition_id, const int64_t* offsets,
                                   const uint16_t* sample_idx, int64_t nv);
int vpca_pool_accumulate_bits(vpca_pool* pool, int64_t partition_id, const uint8_t* bits, int64_t nv, int64_t stride_bytes);
int vpca_pool_accumulate_bed(vpca_pool* pool, int64_t partition_id, const uint8_t* rows, int64_t nv, int64_t stride_bytes,
                             int32_t counted_allele);
int vpca_pool_commit(vpca_pool* pool, int64_t partition_id);
int vpca_pool_abort(vpca_pool* pool, int64_t partition_id);
int vpca_pool_reduce_and_finalize(vpca_pool* pool);
int vpca_pool_get_gram(vpca_pool* pool, int32_t* out);
int vpca_pool_compute_pca(vpca_pool* pool, int32_t k, double* vecs, double* evals, int32_t* non_zero_rows);
/* Sum of the per-GPU statistics (times: the maximum). */
struct vpca_stats;
int vpca_pool_get_stats(vpca_pool* pool, struct vpca_stats* out);

/* ---- synthetic cohort (stands in for the retired Genomics API ingestion, rdd/VariantsRDD.scala:187-236;
 *      specification in DESIGN.md "Synthetic generator") --------------------------------------------------
 * Fill a dense sample-major device tile d_x[s * ld + (v - v0)] for variants [v0, v0+nv).
 * mode 0: binary carrier x = (dosage > 0) (reference encode rule); mode 1: dosage 0/1/2. */
int vpca_synth_dense_device(vpca_ctx* ctx, uint64_t seed, int64_t v0, int64_t nv, int mode, void* d_x, int64_t ld);

/* Same generator, writing the panel layout of vpca_accumulate_panels (buffer: ceil(nv / P) * n_samples * P cells). */
int vpca_synth_panels_device(vpca_ctx* ctx, uint64_t seed, int64_t v0, int64_t nv, int mode, void* d_x,
                             int64_t panel_variants);

/* ---- introspection ---------------------------------------------------------------------------------- */
typedef struct vpca_stats {
    int64_t variants_accumulated; /* rows folded into the Gram or into staged partitions                  */
    int64_t gram_launches;        /* tcgen05 Gram kernel launches                                         */
    int64_t kernel_launches;      /* all kernels launched by this ctx                                     */
    int64_t h2d_bytes;            /* bytes copied host -> device by accumulate_* / encode / set_gram      */
    int64_t d2h_bytes;            /* bytes copied device -> host by get_* / compute_pca                   */
    float last_gram_ms;           /* device time of the most recent Gram launch (CUDA events)             */
    float last_eig_ms;            /* device time of the most recent centering + eigensolve                */
    int32_t gram_cta_group;       /* 1 or 2: tcgen05 cta_group used                                       */
    int32_t gram_resident;        /* 1 when the last launch kept accumulators in TMEM for the whole K loop */
    int32_t eig_method;           /* last vpca_compute_pca: 1 direct reduction, 2 Lanczos, 3 Lanczos abandoned -> direct */
    int32_t eig_iterations;       /* Lanczos steps taken by the last vpca_compute_pca (0 for a direct solve)  */
} vpca_stats;
int vpca_get_stats(vpca_ctx* ctx, vpca_stats* out);
/* Diagnostic (set VPCA_GRAM_PROF=1 before the first Gram launch): per-CTA timestamps of the last Gram launch,
 * 4 x int64 nanoseconds per CTA {start, -, last MMA issued, end}; returns the number of CTAs written (<= max_ctas)
 * or a negative vpca_status.  Synchronises the stream. */
int vpca_debug_gram_profile(vpca_ctx* ctx, int64_t* out, int32_t max_ctas);
/* Diagnostic (set VPCA_LZ_PROF=1 before the first vpca_compute_pca): block 0's timestamps of the persistent Lanczos kernel,
 * 8 x int64 nanoseconds per step {step start, start vector staged + norms, mat-vec done, y and the new basis column written,
 * shares of V^T y and V^T v_j written, first grid barrier passed, fused Gram-Schmidt pass done, next start vector written
 * (second grid barrier next)}
 * for steps 0..31 (each slot holds the last launch that ran that step index); returns the number of steps written or a
 * negative vpca_status. */
int vpca_debug_lanczos_profile(vpca_ctx* ctx, int64_t* out, int32_t max_steps);

/* ---- Multi-dataset keying on the device (SURVEY 8 f-3) ------------------------------------------------------------
 * The 2-dataset and N-dataset branches of VariantsPcaDriver.getCallsRdd (VariantsPca.scala:153-168) key every variant by
 * getVariantKey (:62-78: Guava Hashing.murmur3_128() over contig, start, end, reference bases, alternate bases) and then
 * join (:115-128) or merge (:136-148) the datasets on that key.  Here the rows of ALL datasets are handed over as one CSR
 * (rows of dataset 0 first) next to the key bytes of every row; hashing, the hash join / group-by and the concatenation
 * of the calls run on the GPU, and the joined rows can be accumulated without leaving it.
 *
 * vpca_hash_keys: MurmurHash3_x64_128 (seed 0) of nkeys byte strings, key q = payload[key_offsets[q], key_offsets[q+1]);
 *   out[2q], out[2q+1] = the two little-endian 64-bit halves of Guava's HashCode.asBytes() (HashCode.toString is their
 *   bytes in hex).  Host buffers in and out.
 * vpca_join_rows: mode VPCA_JOIN -- rows [0, n_left) are the left dataset, rows [n_left, nrows) the right one; one
 *   output row per (left, right) pair with equal keys, left calls then right calls (`related._1 ++ related._2`, :127),
 *   ordered by left row, then right row.  mode VPCA_MERGE -- n_left is ignored; keys that occur exactly
 *   variant_set_count times (:144) yield one row: the calls of the group's rows in input order (:145), rows ordered by
 *   the group's first input row.  sample_idx holds the calls that survive `_.hasVariation` (:164), already mapped to
 *   [0, n_samples).  The result stays on the device inside the context until the next vpca_join_rows / vpca_reset;
 *   *out_rows / *out_nnz report its size.  Driver-side step (the reference's join is a shuffle stage that precedes the
 *   mapPartitions tasks): one join at a time per context.
 * vpca_join_fetch: copies the retained result to the host (out_offsets: out_rows + 1, out_idx: out_nnz entries).
 * vpca_accumulate_joined: encodes the retained rows and accumulates them into the staging Gram of partition_id, exactly
 *   like vpca_accumulate_calls would for the same rows (commit / abort as usual); no host round trip of the joined rows. */
#define VPCA_JOIN 0
#define VPCA_MERGE 1
int vpca_hash_keys(vpca_ctx* ctx, const uint8_t* payload, const int64_t* key_offsets, int64_t nkeys, uint64_t* out);
int vpca_join_rows(vpca_ctx* ctx, int32_t mode, int32_t variant_set_count, int64_t n_left, const uint8_t* key_payload,
                   const int64_t* key_offsets, const int64_t* offsets, const int32_t* sample_idx, int64_t nrows,
                   int64_t* out_rows, int64_t* out_nnz);
int vpca_join_fetch(vpca_ctx* ctx, int64_t* out_offsets, int32_t* out_idx);
/* rows / calls of the retained result (what vpca_join_fetch will write); VPCA_ERR_STATE when there is none */
int vpca_join_size(vpca_ctx* ctx, int64_t* out_rows, int64_t* out_nnz);
int vpca_accumulate_joined(vpca_ctx* ctx, int64_t partition_id);

/* Host-only introspection of the Gram schedule (works without a GPU; what tests/test_schedule.py checks).
 * vpca_debug_tiles: the output tiles the kernel enumerates for n_samples -- 8 int32 per tile {rowA of CTA 0, rowA of CTA 1,
 *   rowB, n_eff (MMA N), weight prefix, flags (1: a 128-block above the diagonal is written transposed, 2: CTA 1 is a
 *   filler), 0, 0}; exact != 0: the exact 128-block cover of the lower triangle (every block of
 *   `for (c1 <- callset; c2 <- callset)`, VariantsPca.scala:186-188, with c2 <= c1 computed exactly once), 0: the 256 x 240
 *   rectangles kind::mxf4 uses.  Returns the tile count (may exceed max_tiles).
 * vpca_debug_plan: the (worker, tile, first k-block, end k-block, TMEM column, TMEM columns of the worker) pieces of one
 *   window of kb_window k-blocks under an equal split -- 6 int32 per piece; returns the piece count, or -(1 + worker) when
 *   a worker would own more pieces than the kernel supports.
 * vpca_debug_rebalance: what the on-device rebalancer does with a candidate speed-weighted split before it publishes it --
 *   `cum` (workers + 1 fractions of a window, cum[0] = 0, cum[workers] = 1; in / out) is repaired so that the accumulators
 *   of every worker fit `col_limit` TMEM columns (512; 480 for kind::mxf4), then the pieces are written like
 *   vpca_debug_plan.  Returns the piece count, or VPCA_ERR_STATE when no repair exists (the device keeps the old split). */
int vpca_debug_rebalance(const int32_t* tiles, int32_t num_tiles, int32_t workers, int32_t kb_window, int32_t col_limit,
                         double* cum, int32_t* out, int32_t max_pieces);
int vpca_debug_tiles(int32_t n_samples, int32_t cta_group, int32_t exact, int32_t* out, int32_t max_tiles);
/* Host-only: the tiles (int8 / bf16 rectangles, same 8-int records as vpca_debug_tiles) an owner-computes context that
 * stores rows [row0, row0 + rows) of the Gram enumerates -- only products whose rows of S lie in the band. */
int vpca_debug_band_tiles(int32_t n_samples, int32_t cta_group, int32_t row0, int32_t rows, int32_t* out, int32_t max_tiles);
/* Diagnostic: how many clusters of cluster_size CTAs of the Gram kernel (one CTA per SM) `device` can hold at once
 * (cudaOccupancyMaxActiveClusters); negative vpca_status on error. */
int vpca_debug_max_clusters(int32_t device, int32_t cluster_size);
int vpca_debug_plan(const int32_t* tiles, int32_t num_tiles, int32_t workers, int32_t kb_window, int32_t* out, int32_t max_pieces);

#ifdef __cplusplus
}
#endif
#endif /* VPCA_H_ */

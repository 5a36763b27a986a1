/*
 * ise.h -- C ABI of libise.so, the B200 (sm_100a) retrieval core that replaces the
 * Faiss-CPU / NumPy arithmetic behind image-search-engine's hot path.
 *
 * The reference (ManuelZ/image-search-engine) has no FFI of its own: its hot path is
 * Python calling the third-party `faiss` module.  Each entry point below names the
 * reference call site (file:line under /root/reference/backend) whose arithmetic it
 * replaces; INTEGRATION.md shows the ctypes binding a maintainer adds on the
 * reference side.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; ise_last_error() returns
 *     a thread-local message for the last failing call on this thread;
 *   - all data pointers are DEVICE pointers owned by the caller unless the parameter is
 *     documented as host memory; the library never allocates result memory, scratch is
 *     sized by the matching *_workspace_bytes() call;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - row-major, float32 unless stated; ids are int64 like Faiss idx_t;
 *   - no global mutable state besides the per-device ise_ctx.
 */
#ifndef ISE_H_
#define ISE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ISE_VERSION 100

/* faiss MetricType values (faiss/MetricType.h): inner product = 0, L2 = 1 */
#define ISE_METRIC_IP 0
#define ISE_METRIC_L2 1

/* element type of raw descriptor rows (descriptors.py:216-258: ORB/BRISK uint8, SIFT float32) */
#define ISE_DTYPE_F32 0
#define ISE_DTYPE_U8 1
/* rows of an FP16 hi plane written by ise_prepare_rows (ise_kmeans_accumulate_sorted only) */
#define ISE_DTYPE_F16 2

/* histogram binning: np.histogram(idx, bins=k) over [min,max] (bag_of_visual_words.py:103,
 * SURVEY quirk Q1) or the intended bincount(idx, minlength=k) */
#define ISE_HIST_NUMPY_COMPAT 0
#define ISE_HIST_BINCOUNT 1

/* output element type of the histogram matrix (reference: float64, bag_of_visual_words.py:100) */
#define ISE_OUT_F32 0
#define ISE_OUT_F64 1

typedef struct ise_ctx ise_ctx;

/* ---- context / errors ---------------------------------------------------------------- */
int ise_version(void);
const char* ise_last_error(void);
/* device = CUDA ordinal; fails (no CPU fallback) when no sm_100 device is present */
int ise_ctx_create(int device, ise_ctx** out);
void ise_ctx_destroy(ise_ctx* ctx);
int ise_ctx_sm_count(const ise_ctx* ctx);

/* ---- host-side helpers (pure CPU, sequential RNG semantics of Faiss) ------------------ */
/* faiss::rand_perm(perm, n, seed) restricted to its first m entries (Clustering.cpp
 * subsample_training_set + centroid init; reached from kmeans_faiss.py:41).  out: HOST int64[m]. */
int ise_rand_perm_prefix(int64_t n, int64_t seed, int64_t m, int64_t* out_host);
/* faiss Clustering.cpp split_clusters(): given HOST hassign[k] (modified in place) computes the
 * ordered list of (empty ci, donor cj) pairs with RandomGenerator(1234).  pairs_host: int32[2*k].
 * Returns the number of splits in *nsplit. */
int ise_split_plan(float* hassign_host, int64_t k, int64_t n, int32_t* pairs_host, int32_t* nsplit);
/* split_clusters re-seeds mt19937(1234) on every call, so libise keeps a process-wide sparse index of that stream
 * (the draws small enough to ever accept a donor); this starts generating its first n_draws entries in a background
 * thread and returns at once.  Optional: ise_split_plan extends the index itself when it runs past it. */
int ise_split_plan_warm(int64_t n_draws);

/* Ragged ingestion (pure CPU, multi-threaded): the reference's input contract is a Python list with one (n_i, d)
 * row-major array per image (descriptors.py:104-139), concatenated by one single-threaded np.concatenate
 * (bag_of_visual_words.py:128).  Copies images [i0, i1) -- srcs[i] = HOST pointer of image i, offsets[n_img + 1] =
 * cumulative row counts -- to dst_base + offsets[i] * d * sizeof(dst element), i.e. straight into the caller's (pinned)
 * packed matrix.  src F32 -> dst U8 narrows on the way and sets *ok = 0 (dst undefined) unless every value is an
 * integer in [0, 255] (OpenCV SIFT / ORB-as-float descriptors are): a quarter of the host -> device bytes. */
int ise_pack_rows(const void* const* srcs_host, const int64_t* offsets_host, int64_t i0, int64_t i1, int d,
                  int src_dtype, int dst_dtype, void* dst_base_host, int nthreads, int* ok);
/* The same copy as a background job over n_chunks consecutive image ranges [image_cuts[c], image_cuts[c + 1]): the
 * worker threads finish the chunks IN ORDER, so the caller sends chunk c to the device (ise_pack_wait(job, c, &ok)
 * returns once its rows are in place; ok = 0: some value did not fit uint8, start over in float32) while chunk c + 1
 * is still being packed.  srcs / offsets / dst stay valid until ise_pack_end, which joins the threads. */
int ise_pack_begin(const void* const* srcs_host, const int64_t* offsets_host, const int64_t* image_cuts, int n_chunks,
                   int d, int src_dtype, int dst_dtype, void* dst_base_host, int nthreads, void** job);
int ise_pack_wait(void* job, int chunk, int* ok);
/* Two-ended use (a caller that can also send a chunk in its source format): ise_pack_poll is the non-blocking form of
 * ise_pack_wait (done = 1: the workers have finished the chunk); ise_pack_claim takes a chunk the workers have not
 * started away from them (claimed = 1: they will skip it) -- the workers walk the chunks from the front, the caller
 * claims from the back whenever its copy engine is idle, and the two meet where host and PCIe bandwidth balance. */
int ise_pack_poll(void* job, int chunk, int* done, int* ok);
int ise_pack_claim(void* job, int chunk, int* claimed);
int ise_pack_end(void* job);

/* ---- operand preparation --------------------------------------------------------------
 * The distance contractions run on the tcgen05 tensor cores as FP16 "hi + lo" split
 * products (hi*hi + hi*lo + lo*hi, FP32 accumulate) which carries ~22-24 mantissa bits:
 * rows are scaled by a per-tensor power of two, hi = fp16(s*x), lo = fp16(s*x - hi).
 * meta (device float[8]) = { scale, 1/scale, lo_nonzero (0/1), absmax, max row norm^2, 0, 0, 0 }.
 * ldp (elements) = row pitch of the planes, multiple of 8, >= d; pad columns are zeroed.
 * norms (nullable) = exact FP32 sum of squares per row (fvec_norms_L2sqr).
 * Replaces: the implicit float32 conversion `X.astype(np.float32)` + Faiss's internal
 * operand packing for sgemm (kmeans_faiss.py:41,49; utils.py:327 index.add). */
int ise_prepare_planes(ise_ctx* ctx, const void* x, int dtype, int64_t n, int d, int64_t ldx,
                       void* hi, void* lo, int64_t ldp, float* norms, float* meta, void* stream);

/* ROW operands (descriptor rows of an assign, query rows of a search) in ONE pass over x: every row gets its own
 * power-of-two scale (row_inv[n] = 1 / scale; meta's scale fields are 1), so no absmax pre-pass is needed -- the
 * selection epilogue owns one row per thread and rescales its accumulator by that row's factor.  Rows whose lo part is
 * all zero skip the lo store (lo_skipped[n]: device scratch bytes, required when lo != NULL).  meta[7] != 0 reports
 * NaN / Inf in x (faiss.Kmeans.train refuses such input, kmeans_faiss.py:41).  Pass row_inv as a_row_inv to
 * ise_gemm_select / ise_gemm_collect / ise_rescore_select.  Replaces the host-side `X.astype(np.float32)` of
 * kmeans_faiss.py:41,49 for the row side. */
int ise_prepare_rows(ise_ctx* ctx, const void* x, int dtype, int64_t n, int d, int64_t ldx,
                     void* hi, void* lo, int64_t ldp, float* norms, float* row_inv, uint8_t* lo_skipped,
                     float* meta, void* stream);

/* One read-only pass over a float32 matrix: meta[3] = max |x|, meta[7] != 0 when it holds a NaN or an Inf (Faiss's
 * Clustering::train validates ALL of its input before sub-sampling it, kmeans_faiss.py:41). */
int ise_scan_f32(ise_ctx* ctx, const float* x, int64_t n, int d, int64_t ldx, float* meta, void* stream);

/* faiss.normalize_L2 (utils.py:303, engine.py:53, siamese/test_index.py:53): in place,
 * x *= 1/sqrtf(sum x^2) for rows with non-zero norm. */
int ise_normalize_l2(ise_ctx* ctx, float* x, int64_t n, int d, void* stream);

/* ---- fused distance contraction + selection (the hot kernel) ---------------------------
 * For every row r of A (m rows) selects the topk best columns of B (n rows) under
 *   IP : score = <a_r, b_c>                  best = largest   (IndexFlatIP.search)
 *   L2 : score = |a_r|^2 + |b_c|^2 - 2<a,b>  best = smallest, clamped at 0 (IndexFlatL2.search)
 * without ever writing the m x n score matrix to HBM.  Ties: lower id wins.
 * Output rows are sorted best-first; when topk > n the tail is id -1 / -+FLT_MAX like Faiss.
 * a_lo / b_lo may be NULL when the corresponding meta says lo_nonzero == 0 (exact operand).
 * a_norms / b_norms are required for L2 only.  out ids = column + id_base.
 * a_row_inv (nullable): per-row 1 / scale of the A planes from ise_prepare_rows (overrides a_meta's scale).
 * row_seed (nullable, topk > 1): per-row score of a column known to exist (IP score / L2 distance, e.g. the
 * best hit in a column sample); only columns strictly better than it are kept, so lists may come back
 * shorter than topk (padded with id -1).  It removes nearly all selection traffic from the epilogue.
 * flag_rows / flag_count (nullable, topk == 1, unsplit column range, a_norms required): coarse top-1
 * verification.  Called with the hi planes only (a_lo = b_lo = NULL) the kernel also tracks the exact
 * runner-up score of every row and appends to flag_rows[0 .. *flag_count) the rows whose winner is not
 * separated from the runner-up by more than the rigorous coarse error bound (CoarseBound, common.cuh);
 * the caller re-runs just those rows with the lo planes.  All other rows are provably correct.
 * Replaces index.search inside faiss.Kmeans.train (kmeans_faiss.py:41), FaissKMeans.transform
 * (kmeans_faiss.py:49) and run_image_query (engine.py:55) / query_index (siamese/test_index.py:54). */
size_t ise_gemm_select_workspace_bytes(ise_ctx* ctx, int64_t m, int64_t n, int d, int topk);
int ise_gemm_select(ise_ctx* ctx,
                    const void* a_hi, const void* a_lo, int64_t lda, const float* a_meta, const float* a_norms,
                    const float* a_row_inv,
                    const void* b_hi, const void* b_lo, int64_t ldb, const float* b_meta, const float* b_norms,
                    int64_t m, int64_t n, int d, int metric, int topk, int64_t id_base,
                    const float* row_seed, int32_t* flag_rows, int32_t* flag_count,
                    float* out_val, int64_t* out_idx,
                    void* workspace, size_t workspace_bytes, void* stream);

/* FUSED ASSIGN (top-1): takes the RAW float32 rows x[m, d] and converts them inside the contraction kernel -- four extra
 * warps per CTA turn the rows of the CTA's NEXT work item into per-row-scaled FP16 planes (the ise_prepare_rows method)
 * while the tensor pipe works on the current one, so the HBM-bound preparation pass disappears behind the MMAs.  The
 * row operand comes out as a by-product (a_hi / a_lo planes with pitch lda, a_norms, a_row_inv, a_meta: the same
 * contents ise_prepare_rows writes), ready for ise_rescore_topk / ise_kmeans_accumulate_sorted.  Only the hi plane of
 * A is multiplied in the fused launch; when the rows turn out NOT to be exact in it (a_meta[2] != 0, decided on the
 * device) the lo plane is completed and the assign repeated with it by two follow-up launches that return at once
 * otherwise -- keypoint descriptors (integer SIFT, ORB / BRISK as float) are exact.  a_lo may be NULL only when the
 * caller knows that (no repeat pass then).  Returns 2 and does nothing when the shape is not covered (d % 4 != 0,
 * d > 128, unaligned rows, or too few rows for an unsplit column range): run ise_prepare_rows + ise_gemm_select then.
 * Replaces `X.astype(np.float32)` + index.search(X, 1) of FaissKMeans.transform (kmeans_faiss.py:49). */
int ise_assign_fused(ise_ctx* ctx, const float* x, int64_t ldx, int64_t m, int d,
                     void* a_hi, void* a_lo, int64_t lda, float* a_norms, float* a_row_inv, uint8_t* a_lo_skipped,
                     float* a_meta,
                     const void* b_hi, const void* b_lo, int64_t ldb, const float* b_meta, const float* b_norms,
                     int64_t n, int metric, int64_t id_base, float* out_val, int64_t* out_idx,
                     void* workspace, size_t workspace_bytes, void* stream);

/* VERIFIED ASSIGN (d <= 128): quantisation and the k-means assign need the nearest column's ID, and an id only needs
 * ONE tensor-core product per tile plus a proof.  With workspace != NULL (ise_assign_workspace_bytes) ise_assign_fused
 * -- and ise_assign_verified, the same pipeline over PREPARED row planes (k-means iterations prepare the rows once) --
 * runs: (1) a one-product pass (hi planes) whose epilogue tracks the exact runner-up of every row and lists the rows
 * whose winner is not separated from it by more than twice the rigorous error bound of the neglected lo-plane /
 * accumulation terms; the 128-row tile of a work item stays resident in shared memory and only B streams; (2) a
 * compaction of the listed rows' planes; (3) the split products over the compacted rows, row count read on the device,
 * results scattered back; (4) a launch that repeats everything with the split products and returns at once unless the
 * list overflowed its capacity (a quarter of the rows).  No host synchronisation anywhere.  Ids are those of the split
 * products; out_val holds one-product scores (|error| <= the bound) for the rows decided in (1) -- callers that need
 * distances pass workspace = NULL or re-score (ise_rescore_topk).  workspace[0..2] (int32) afterwards: listed rows, rows
 * re-run, overflow flag.  Both return 2 (nothing done; ise_assign_fused falls back to its plain mode by itself) when
 * the shape is not covered: d > 128, fewer than 8 stages of B per row tile, or too few rows to fill the machine with an
 * unsplit column range.  Replaces index.search(X, 1) of FaissKMeans.transform (kmeans_faiss.py:49) and the assign of
 * faiss.Kmeans.train (kmeans_faiss.py:41). */
size_t ise_assign_workspace_bytes(ise_ctx* ctx, int64_t m, int d);
int ise_assign_verified_covers(ise_ctx* ctx, int64_t m, int64_t n, int d);   /* 1 = the verified pipeline takes this shape */
int ise_assign_verified(ise_ctx* ctx,
                        const void* a_hi, const void* a_lo, int64_t lda, const float* a_meta, const float* a_norms,
                        const float* a_row_inv,
                        const void* b_hi, const void* b_lo, int64_t ldb, const float* b_meta, const float* b_norms,
                        int64_t m, int64_t n, int d, int metric, int64_t id_base,
                        float* out_val, int64_t* out_idx, void* workspace, size_t workspace_bytes, void* stream);

/* COLLECT variant of the fused contraction for large k: instead of keeping a bounded list per row, every
 * column whose (coarse) score beats row_seed[row] is appended to the row's buffer cand_*[row, 0..cap)
 * (unsorted; row_count[row] = number of qualifying columns, which may exceed cap = overflow; unused slots
 * hold id -1).  ise_rescore_select(row_count=...) then sorts and proves the top-k.  Same operand rules as
 * ise_gemm_select. */
int ise_gemm_collect(ise_ctx* ctx,
                     const void* a_hi, const void* a_lo, int64_t lda, const float* a_meta, const float* a_norms,
                     const float* a_row_inv,
                     const void* b_hi, const void* b_lo, int64_t ldb, const float* b_meta, const float* b_norms,
                     int64_t m, int64_t n, int d, int metric, int64_t id_base, const float* row_seed, int cap,
                     float* cand_val, int64_t* cand_idx, int32_t* row_count, void* stream);

/* Exact FP32 CUDA-core path for small query counts: Faiss computes n < 20 queries without the
 * BLAS expansion (distances.cpp exhaustive_*_seq: direct dot / sum (x-y)^2), which is what the
 * reference's single-image query hits (engine.py:55 with nq = 1).  Also used as the on-device
 * cross-check of the tensor-core path in tests.  q, db: FP32 rows. */
size_t ise_flat_search_exact_workspace_bytes(ise_ctx* ctx, int64_t nq, int64_t nb, int topk);
int ise_flat_search_exact(ise_ctx* ctx, const float* q, int64_t nq, const float* db, int64_t nb, int d,
                          int metric, int topk, int64_t id_base, float* out_val, int64_t* out_idx,
                          void* workspace, size_t workspace_bytes, void* stream);

/* The two stages of ise_flat_search_exact on their own, for k > 128 (Faiss's IndexFlat.search takes any k,
 * engine.py:55): scores[nq, nb] = direct FP32 <q,y> / sum (q-y)^2 of every pair; ise_scores_mask overwrites the entries a
 * selection pass returned (idx[nq, kk], -1 = padding) with -+inf so that the next ise_scores_topk pass yields the next
 * best kk in the same canonical (score, id) order. */
int ise_pair_scores(ise_ctx* ctx, const float* q, int64_t nq, const float* db, int64_t nb, int d, int metric,
                    float* scores, void* stream);
int ise_scores_mask(ise_ctx* ctx, float* scores, int64_t nq, int64_t nb, const int64_t* idx, int kk,
                    int64_t id_base, int metric, void* stream);

/* Exact FP32 re-score + re-rank of already selected candidates (CUDA cores).  The tensor-core
 * accumulator truncates, which shows in returned distances (not in which candidates are picked); this
 * recomputes val[m,topk] for the ids in idx[m,topk] from the original rows with Faiss's formulas
 * (IP: <a,b>;  L2: max(0, |a|^2 + |b|^2 - 2<a,b>), distances.cpp) and re-sorts each row by (score, id).
 * a: [m,d] f32 or u8 rows, b: [n,d] f32 rows, ids are global (= column + id_base), -1 = padding. */
int ise_rescore_topk(ise_ctx* ctx, const void* a, int a_dtype, int64_t lda, const float* b, int64_t ldb,
                     int64_t m, int64_t n, int d, int metric, int topk, int64_t id_base,
                     const float* a_norms, const float* b_norms, float* val, int64_t* idx, void* stream);

/* Coarse-then-verify search: `cand_*` [m, kc] are the kc best columns per row found by a COARSE
 * ise_gemm_select call (hi planes only: pass a_lo = b_lo = NULL, one tcgen05 product instead of three).
 * This kernel re-scores all kc candidates exactly in FP32, writes the exact top-k [m, topk] and PROVES
 * per row that no column outside the candidate list can belong to the top-k, using the rigorous bound
 * |coarse - exact| <= kappa |a| max|b| (kappa from the FP16 rounding of the planes + accumulator
 * truncation, see rescore.cu).  Rows that cannot be proven are appended to flag_rows[0 .. *flag_count)
 * (device int32) and must be re-run by the caller with the full-precision split products.
 * row_seed (nullable): the seed the coarse call was given; it then also bounds the unseen columns.
 * row_count (nullable): candidates come from ise_gemm_collect (unsorted, kc = cap <= 1024). */
int ise_rescore_select(ise_ctx* ctx, const void* a, int a_dtype, int64_t lda, const float* a_meta,
                       const float* a_norms, const float* a_row_inv, const float* b, int64_t ldb, const float* b_meta,
                       const float* b_norms, int64_t m, int64_t n, int d, int metric, int kc, int topk,
                       int64_t id_base, const float* row_seed, const int32_t* row_count,
                       const float* cand_val, const int64_t* cand_idx,
                       float* out_val, int64_t* out_idx, int32_t* flag_rows, int32_t* flag_count, void* stream);

/* ---- range search over the flat index (faiss/IndexFlat.cpp IndexFlat::range_search ->
 * faiss/utils/distances.cpp range_search_inner_product / range_search_L2sqr) ------------------------------
 * Every column whose exact FP32 score beats `radius` (IP: dis > radius, L2: squared dis < radius; strict).
 * Results of a row are in ascending id.  Tensor-core path (nq >= 20), no host round trip inside a step:
 *   ise_range_seed:  row_seed[m] for ise_gemm_collect = radius loosened by the rigorous coarse bound of the hi-plane
 *                    product (eps for IP, 2 eps for L2) plus the FP32 re-score's rounding and a few ulps, so that the
 *                    collect over hi-only planes appends EVERY column whose exact score can qualify.  Operands and
 *                    their meta / norms / row_inv as prepared for the collect (a_row_inv nullable).
 *   ise_gemm_collect (unchanged; hi planes only, cap slots per row);
 *   ise_range_count: exact FP32 re-score of the first min(row_count, cap) candidates of every row (rescore formulas:
 *                    <a,b>, or max(0, |a|^2 + |b|^2 - 2<a,b>)); passes get the exact score in cand_val, failures id -1
 *                    in cand_idx.  kept[m + 1] int64: kept per row, 0 for overflowing rows (row_count > cap: the
 *                    caller re-runs them with a larger cap), kept[m] = 0.  a: f32 or u8 rows, b: f32 rows.
 *   ise_range_lims:  lims[m + 1] = base + exclusive scan of kept[m + 1].
 *   ise_range_fill:  kept pairs of candidate row i -> out[lims[row_map ? row_map[i] : i] ...] (slot order); rows with
 *                    row_count > cap are skipped.
 *   ise_range_sort:  sorts every segment [lims[r], lims[r+1]) of (ids, dis) by id, in place (lims[0] = 0,
 *                    total < 2^31). */
int ise_range_seed(ise_ctx* ctx, const float* a_meta, const float* a_norms, const float* a_row_inv,
                   const float* b_meta, int64_t m, int d, int metric, float radius, float* row_seed, void* stream);
int ise_range_count(ise_ctx* ctx, const void* a, int a_dtype, int64_t lda, const float* b, int64_t ldb,
                    int64_t m, int64_t n, int d, int metric, float radius, int64_t id_base,
                    const float* a_norms, const float* b_norms, int cap, const int32_t* row_count,
                    float* cand_val, int64_t* cand_idx, int64_t* kept, void* stream);
size_t ise_range_lims_workspace_bytes(ise_ctx* ctx, int64_t m);
int ise_range_lims(ise_ctx* ctx, const int64_t* kept, int64_t m, int64_t base, int64_t* lims,
                   void* workspace, size_t workspace_bytes, void* stream);
int ise_range_fill(ise_ctx* ctx, int64_t m, int cap, const int32_t* row_count, const float* cand_val,
                   const int64_t* cand_idx, const int64_t* row_map, const int64_t* lims, float* out_dis,
                   int64_t* out_ids, void* stream);
size_t ise_range_sort_workspace_bytes(ise_ctx* ctx, int64_t m, int64_t total);
int ise_range_sort(ise_ctx* ctx, int64_t m, const int64_t* lims, int64_t total, float* dis, int64_t* ids,
                   void* workspace, size_t workspace_bytes, void* stream);
/* Exact path (nq < 20, Faiss's direct per-pair formulas): range search over scores[nq, nb] of ise_pair_scores.
 * Writes lims[nq + 1] (= base + offsets) always and, when out_dis / out_ids are given (length lims[nq] - base),
 * the qualifying (score, id_base + column) pairs in column order. */
size_t ise_scores_range_workspace_bytes(ise_ctx* ctx, int64_t nq, int64_t nb);
int ise_scores_range(ise_ctx* ctx, const float* scores, int64_t nq, int64_t nb, int metric, float radius,
                     int64_t id_base, int64_t base, int64_t* lims, float* out_dis, int64_t* out_ids,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Merge g sorted top-k lists per row ([g, m, topk] each) into one; canonical (score, id) order.
 * Used for column-split partial results and for the cross-GPU merge of a sharded index. */
int ise_topk_merge(ise_ctx* ctx, const float* val_parts, const int64_t* idx_parts, int g, int64_t m,
                   int topk, int metric, float* out_val, int64_t* out_idx, void* stream);

/* ---- k-means centroid update (faiss Clustering.cpp compute_centroids / split_clusters /
 * post_process_centroids, reached from kmeans_faiss.py:41) ------------------------------- */
/* sums[k,d] += x rows by assignment, counts[k] += 1 (float, like hassign), obj[0] += sum of the rows'
 * objective terms: with `centroids` [k,d] given they are recomputed in exact FP32 here (IP: <x,c>,
 * L2: sum (x-c)^2) from the row already in registers, otherwise dis[] is summed.
 * accum buffers must be zeroed by the caller (so several shards / ranks can add into them).
 * k = number of centroids (rows of sums): lets the library tile the sum matrix over the SMs' shared memory
 * (privatised scatter-add) when it is small enough; k <= 0 selects the plain global-atomic kernel. */
int ise_kmeans_accumulate(ise_ctx* ctx, const void* x, int dtype, int64_t n, int d, int64_t ldx,
                          const int64_t* assign, const float* dis, const float* centroids, int64_t k, int metric,
                          float* sums, float* counts, double* obj, void* stream);
/* Same contract, atomics-free: the rows are grouped by centroid with a counting sort (ids -> histogram -> scan ->
 * scatter of (centroid, row) pairs), the sorted list is cut into fixed 64-row chunks and each chunk is gathered with
 * 128-bit loads and summed in registers, one vector reduction per lane per run of equal ids (C2: ~1.3 per 64 rows
 * instead of 64).  dtype ISE_DTYPE_F16: x is the FP16 hi plane of ise_prepare_rows (pitch ldx halves) and row_inv its
 * per-row 1 / scale -- valid when the operand is exact in that plane (meta lo_nonzero == 0: integer-valued SIFT, ORB),
 * and half the gather traffic of the FP32 rows; row_inv is NULL otherwise.
 * Objective always recomputed from `centroids` (nullable: no objective).  Falls back to
 * ise_kmeans_accumulate for rows that are not 4-column aligned.  workspace: ise_kmeans_accumulate_workspace_bytes. */
size_t ise_kmeans_accumulate_workspace_bytes(ise_ctx* ctx, int64_t n, int64_t k);
int ise_kmeans_accumulate_sorted(ise_ctx* ctx, const void* x, int dtype, int64_t n, int d, int64_t ldx,
                                 const float* row_inv,
                                 const int64_t* assign, const float* centroids, int64_t k, int metric,
                                 float* sums, float* counts, double* obj,
                                 void* workspace, size_t workspace_bytes, void* stream);
/* centroids = sums / counts for non-empty clusters (empty rows stay zero); n_empty[0] = #empty */
int ise_kmeans_mean(ise_ctx* ctx, const float* sums, const float* counts, int64_t k, int d,
                    float* centroids, int32_t* n_empty, void* stream);
/* apply the ordered split plan from ise_split_plan (pairs on DEVICE int32[2*nsplit]) */
int ise_kmeans_apply_splits(ise_ctx* ctx, float* centroids, int64_t k, int d,
                            const int32_t* pairs, int32_t nsplit, void* stream);

/* ---- BoVW histogram + Okapi tf (bag_of_visual_words.py:98-106, utils.py:153-202) ------- */
/* words[n] int64 visual-word ids, img_offsets[n_img+1] int64 (image i owns [off[i], off[i+1])).
 * out[n_img, k] counts as f32/f64.  mode NUMPY_COMPAT reproduces np.histogram(idx, bins=k)
 * bit-exactly (float64 edge arithmetic); BINCOUNT is bincount(idx, minlength=k).
 * okapi != 0 fuses OkapiTransformer.transform: tf*k1/(tf*k1 + k2*(1-b+b*dl/avgdl)) with
 * dl = row sum, avgdl = mean dl over this batch when the argument is < 0, else the given value (a batch
 * fed in several launches passes the whole batch's mean); zeros stay zero.  n_words = length of words[] (its
 * ratio to n_img picks the warp-per-image kernel for short images); 0 = unknown. */
int ise_bovw_histogram(ise_ctx* ctx, const int64_t* words, int64_t n_words, const int64_t* img_offsets, int64_t n_img,
                       int k, int mode, int out_dtype, void* out,
                       int okapi, double k1, double k2, double b, double avgdl, void* stream);
/* Same histogram (+ fused Okapi), as a CSR matrix with sorted column indices -- what
 * OkapiTransformer.transform returns (scipy CSR, utils.py:153-202) and what
 * `pipeline.transform(...)` hands to its caller (engine.py:96, bag_of_visual_words.py:181-183): the dense
 * [n_img,k] matrix (97 % zeros) is never materialised.  row_nnz: workspace int32[n_img]; indptr:
 * int32[n_img+1]; indices / data: capacity >= number of words (an upper bound on the non-zeros; the used
 * length is indptr[n_img]).  k <= 12288 (shared-memory counters). */
int ise_bovw_histogram_csr(ise_ctx* ctx, const int64_t* words, const int64_t* img_offsets, int64_t n_img,
                           int k, int mode, int out_dtype, int32_t* row_nnz, int32_t* indptr,
                           int32_t* indices, void* data,
                           int okapi, double k1, double k2, double b, double avgdl, void* stream);
/* OkapiTransformer.transform on an existing dense [n_img,k] matrix, in place (f32 or f64).
 * avgdl < 0 => mean row sum of this batch (utils.py:196).  dl_workspace: device double[n_img + 1]. */
int ise_okapi_tf(ise_ctx* ctx, void* h, int out_dtype, int64_t n_img, int k,
                 double k1, double k2, double b, double avgdl, double* dl_workspace, void* stream);

/* OkapiTransformer.transform on a CSR matrix, O(nnz) (utils.py:153-202 works on X.data exactly like this): data[nnz]
 * float64 in place, indptr int64[n_rows + 1], indices int32[nnz] (needed with idf only).  dl = row sums, avgdl < 0 =>
 * mean dl of this batch.  idf (nullable, double[k]) and norm (0 none, 1 l1, 2 l2) are the OPT-IN corrected tf-idf
 * mode: the reference computes idf in fit (utils.py:119-151) and declares norm="l2" (:112) but applies neither, so
 * the drop-in default passes NULL / 0.  dl_workspace: device double[n_rows + 1]. */
int ise_okapi_csr(ise_ctx* ctx, const int64_t* indptr, const int32_t* indices, double* data, int64_t n_rows,
                  double k1, double k2, double b, double avgdl, const double* idf, int norm,
                  double* dl_workspace, void* stream);
/* dense counterpart of the opt-in mode for the GPU-resident index build: h[i, j] *= idf[j] (nullable), then row
 * normalisation (norm as above), in place on an [n_img, k] f32 / f64 matrix already weighted by ise_okapi_tf */
int ise_tfidf_finish(ise_ctx* ctx, void* h, int out_dtype, int64_t n_img, int k, const double* idf, int norm,
                     void* stream);

/* ---- IVFPQ "cell-probe" index (utils.py:311-325: IndexIVFPQ(IndexFlatL2(d), d, 8, 16, 8), nprobe = 5) ---- */
/* per-query top-k of a device score matrix scores[nq, nb] (IP: largest, L2: smallest; +-inf entries are never
 * selected, short rows are padded with id -1): the selection stage of ise_flat_search_exact on its own */
size_t ise_scores_topk_workspace_bytes(ise_ctx* ctx, int64_t nq, int64_t nb, int topk);
int ise_scores_topk(ise_ctx* ctx, const float* scores, int64_t nq, int64_t nb, int metric, int topk, int64_t id_base,
                    float* out_val, int64_t* out_idx, void* workspace, size_t workspace_bytes, void* stream);
/* out[i] = x[i] - centroids[assign[i]]  (faiss compute_residual_n; IndexIVFPQ by_residual) */
int ise_ivfpq_residual(ise_ctx* ctx, const float* x, int64_t ldx, int64_t n, int d, const float* centroids,
                       const int64_t* assign, float* out, void* stream);
/* asymmetric-distance scan of the probed inverted lists: dist[nq, ntotal] (list-sorted order, pre-filled with
 * +inf by the caller) receives sum_m |(q - c_list)_m - pq[m][code_m]|^2 for every code of every probed list.
 * probes[nq, nprobe] int64 list ids (-1 = none), pq_centroids [M, ksub, d/M], codes [ntotal, M] uint8 sorted by
 * list, list_offsets [nlist+1]. */
int ise_ivfpq_scan(ise_ctx* ctx, const float* q, int64_t nq, int d, const float* coarse_centroids, int64_t nlist,
                   const int64_t* probes, int nprobe, const float* pq_centroids, int M, int ksub,
                   const uint8_t* codes, const int64_t* list_offsets, int64_t ntotal, float* dist, void* stream);

/* ---- collectives for a single-process multi-GPU host (NCCL over NVLink, resolved with dlopen at run time) ----------
 * The two exchange steps of the sharded path (SURVEY section 8e): the per-iteration all-reduce of the k-means
 * [k*d sums | k counts] buffer and the all-gather of per-shard top-k lists before ise_topk_merge.  The Python host
 * uses torch.distributed (one process per GPU) over the same NCCL instead; these are for a host that binds libise
 * directly and drives all GPUs from one process.  devs = CUDA ordinals (NULL: 0 .. ndev-1); bufs / send / recv /
 * streams are arrays with one entry per device of the communicator, in communicator order; calls are asynchronous
 * on the given streams.  The reference has no counterpart (single host process, no GPU). */
typedef struct ise_comm ise_comm;
int ise_comm_init_all(int ndev, const int* devs, ise_comm** out);
void ise_comm_destroy(ise_comm* comm);
int ise_comm_size(const ise_comm* comm);
int ise_allreduce_sum_f32(ise_comm* comm, float* const* bufs, int64_t count, void* const* streams);
int ise_allgather(ise_comm* comm, const void* const* send, void* const* recv, int64_t bytes_per_rank,
                  void* const* streams);

#ifdef __cplusplus
}
#endif
#endif /* ISE_H_ */

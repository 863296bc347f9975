/*
 * knn_b200 - B200-native exact (flat) k-nearest-neighbour engine: C ABI.
 *
 * Drop-in boundary for the one hot path of konstin/knn-for-homology: the calls its Python
 * drivers make into faiss-cpu (SWIG) for flat search.  There is no plugin/FFI registry in
 * the reference; the "operator API" is the faiss Python surface itself, so every entry
 * point below names the faiss call it replaces and the reference call sites
 * (paths relative to /root/reference).  The Python binding a maintainer would add is the
 * ctypes stub in knn-for-homology_b200/knn_b200/_lib.py (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; row-major, C-contiguous matrices;
 *   - every function returns 0 on success, a negative KNN_ERR_* otherwise, and leaves a
 *     message retrievable with knn_last_error() (thread-local);
 *   - "host" entry points take host pointers (pageable or pinned), do their own H2D/D2H
 *     copies and return when the result is in the caller's buffers;
 *   - "_dev" entry points take device pointers of the index's device, enqueue on the
 *     cudaStream_t passed as `stream` (NULL = default stream) and may synchronise it;
 *   - the caller owns all buffers; `add` copies (faiss semantics: the drivers reuse and
 *     mutate their arrays after add, pfam/proteins_search.py:37,49);
 *   - an index is not re-entrant: calls on one index come from one thread at a time (the reference's drivers call
 *     faiss sequentially); searches and adds on DIFFERENT streams are ordered against each other by the library;
 *   - the library is CUDA-only: it fails with KNN_ERR_CUDA when no sm_100 device is
 *     usable; there is no CPU fallback.
 */
#ifndef KNN_B200_H
#define KNN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KNN_METRIC_INNER_PRODUCT 0 /* faiss.METRIC_INNER_PRODUCT (cath/search.py:31) */
#define KNN_METRIC_L2 1            /* faiss.METRIC_L2            (cath/search.py:32) */

#define KNN_OK 0
#define KNN_ERR_INVALID (-1) /* bad argument (NULL, shape, k <= 0, ...) */
#define KNN_ERR_CUDA (-2)    /* CUDA runtime / driver failure, or no usable device */
#define KNN_ERR_MEMORY (-3)  /* device or host allocation failed */
#define KNN_ERR_LIMIT (-4)   /* a documented limit was exceeded (k > KNN_MAX_K, more than 2^31-1 rows in one index) */

#define KNN_MAX_K 2048 /* reference uses k in {5,10,11,13,500,1000,2000} (SURVEY.md section 5) */

/* knn_index_create flags */
#define KNN_FLAG_BF16_STORAGE 1u /* keep only bf16 rows (the bf16 values ARE the database; config C5) */

/* Element type of caller rows (database rows and queries) for the `_typed` entry points.  Protein-language-model
 * embeddings usually come in 16 bits (ProtT5's half-precision model writes fp16, C5's database is bf16); the typed
 * calls read them as they are, without an fp32 copy on the host or the device.
 * Contract: a typed call with fp16 or bf16 rows returns exactly what the same call returns on the rows up-converted to
 * fp32 (float(x), which is exact): the same D and I bits, the same stored rows (reconstruct) and the same shadow format.
 * The kernels convert each element at its load and then run the fp32 arithmetic unchanged, and the error bound of the
 * tensor path is computed from the MEASURED rounding of the up-converted values, never assumed.  D stays float32 and
 * I int64.  An unknown dtype code returns KNN_ERR_INVALID.  The untyped entry points are the KNN_DTYPE_F32 calls. */
#define KNN_DTYPE_F32 0  /* float32 */
#define KNN_DTYPE_F16 1  /* IEEE binary16 */
#define KNN_DTYPE_BF16 2 /* bfloat16 */

typedef struct knn_index knn_index;

/* Message of the last error on the calling thread ("" if none). */
const char* knn_last_error(void);

/* Number of CUDA devices visible (0 if CUDA cannot be initialised). */
int knn_device_count(void);

/* faiss.normalize_L2(x): in-place x[i] *= 1/sqrt(sum x[i]^2), zero rows untouched.
 * Call sites: cath/search.py:19, pfam/proteins_search.py:22, seqvec_search/main.py:31,34,
 * pfam/search.py:18,20, pfam/slices/slices_search.py:18. */
int knn_normalize_l2(float* x, int64_t n, int64_t d, int device);
int knn_normalize_l2_dev(float* x_dev, int64_t n, int64_t d, void* stream);

/* faiss.IndexFlat(d, metric) - cath/search.py:20, pfam/proteins_search.py:24,
 * seqvec_search/main.py:35.  `device` = CUDA ordinal. */
int knn_index_create(knn_index** out, int d, int metric, int device, unsigned flags);
int knn_index_free(knn_index* idx);
/* faiss Index::reset(): drop all rows, keep d/metric. */
int knn_index_reset(knn_index* idx);
/* Optional: pre-size the device storage for n rows in total (avoids regrowth copies). */
int knn_index_reserve(knn_index* idx, int64_t n);

/* index.add(xb) - cath/search.py:22, pfam/proteins_search.py:37, seqvec_search/main.py:39.
 * Appends n rows; ids are the implicit row numbers 0..ntotal-1. */
int knn_index_add(knn_index* idx, int64_t n, const float* x);
int knn_index_add_dev(knn_index* idx, int64_t n, const float* x_dev, void* stream);
/* The same for rows of element type `dtype` (KNN_DTYPE_*).  The host form stages 64 MiB chunks of the caller's
 * bytes (twice the rows per chunk for 16-bit rows), so 16-bit rows cross PCIe at half the bytes.  With
 * KNN_FLAG_BF16_STORAGE bf16 rows are stored as they are; fp16 rows are stored as bf16(float(x)). */
int knn_index_add_typed(knn_index* idx, int64_t n, const void* x, int dtype);
int knn_index_add_typed_dev(knn_index* idx, int64_t n, const void* x_dev, int dtype, void* stream);

int64_t knn_index_ntotal(const knn_index* idx);
int knn_index_d(const knn_index* idx);
int knn_index_metric(const knn_index* idx);

/* index.search(xq, k) -> (D, I) - cath/search.py:24, pfam/proteins_search.py:49,
 * seqvec_search/main.py:45.  D: (nq,k) float32, I: (nq,k) int64, best first (IP: largest,
 * L2: smallest squared distance, computed as |x|^2+|y|^2-2<x,y> clamped at 0).  Equal scores:
 * lower id first.  k > ntotal: tail padded with id -1 and -FLT_MAX (IP) / +FLT_MAX (L2).
 * `id_base` (dev variant) is added to every returned id: a shard of a row-sharded database
 * returns global row numbers. */
int knn_index_search(knn_index* idx, int64_t nq, const float* xq, int64_t k, float* D, int64_t* I);
int knn_index_search_dev(knn_index* idx, int64_t nq, const float* xq_dev, int64_t k, float* D_dev,
                         int64_t* I_dev, int64_t id_base, void* stream);
/* The same for queries of element type `dtype` (KNN_DTYPE_*); any query dtype searches any index.  The host form
 * stages and copies the caller's bytes (pinned caller memory is still DMA'd directly). */
int knn_index_search_typed(knn_index* idx, int64_t nq, const void* xq, int dtype, int64_t k, float* D, int64_t* I);
int knn_index_search_typed_dev(knn_index* idx, int64_t nq, const void* xq_dev, int dtype, int64_t k, float* D_dev,
                               int64_t* I_dev, int64_t id_base, void* stream);

/* Two-phase search for a row-sharded database (new; see DESIGN.md section 6).  Phase 1 runs the
 * tensor-core filter over this shard and writes lower_dev[q], a lower bound of the TRUE k-th best score
 * of query q within the shard (L2: of the key 2<x,y> - |y|^2, larger = closer, exact arithmetic)
 * (-FLT_MAX when the shard cannot offer one), and optionally lower_j_dev[q],
 * the same for the j-th best (1 <= j <= k; pass NULL to skip).  The caller combines the bounds of all G
 * shards - element-wise MAX of lower, and with j = ceil(k / G) element-wise MIN of lower_j (every shard holds
 * j rows at or above it, G*j >= k in total), e.g. two NCCL all-reduces - takes the larger of the two and
 * passes it to phase 2, which rescores only the candidates that can still be in the global top-k and returns
 * this shard's (D, I).  At most 131072 queries per call; filter and finish must be called in pairs with the
 * same nq, xq_dev and k.  Scores are comparable across shards for both metrics. */
int knn_index_search_filter_dev(knn_index* idx, int64_t nq, const float* xq_dev, int64_t k, float* lower_dev, int64_t j,
                                float* lower_j_dev, void* stream);
int knn_index_search_finish_dev(knn_index* idx, int64_t nq, const float* xq_dev, int64_t k, const float* lower_dev,
                                float* D_dev, int64_t* I_dev, int64_t id_base, void* stream);
/* Typed forms (queries of element type `dtype`); finish must name the same dtype as filter. */
int knn_index_search_filter_typed_dev(knn_index* idx, int64_t nq, const void* xq_dev, int dtype, int64_t k,
                                      float* lower_dev, int64_t j, float* lower_j_dev, void* stream);
int knn_index_search_finish_typed_dev(knn_index* idx, int64_t nq, const void* xq_dev, int dtype, int64_t k,
                                      const float* lower_dev, float* D_dev, int64_t* I_dev, int64_t id_base,
                                      void* stream);

/* The same two-phase search batch by batch, so that the caller can overlap the exchange + finish of one query batch
 * with the filter of the next on a second stream (knn_b200/distributed.py does: filter of batch b on the main stream,
 * event, then on a side stream all-reduce of that batch's bounds and finish_batch).
 *   begin         fixes (nq, xq_dev, k) - xq_dev must stay valid until `end` - and returns the number of query batches
 *                 and the rows per batch (the last batch may be shorter).  Both depend on nq and the index's
 *                 query_batch alone - batch_rows = min(query_batch, nq) rounded up to 256 - never on the shard's size
 *                 or path, so shards with the same query_batch report identical values and exchange bounds batch by
 *                 batch (an exact-path shard offers no bound and finishes each batch with the exact scan);
 *   filter_batch  filters batch b and writes its bounds into bounds_dev, a caller-zeroed float array
 *                 [nbatches][2][batch_rows]: [b][0][i] = lower bound of the k-th best true score of query
 *                 b*batch_rows+i in this shard, [b][1][i] = MINUS the bound on the j-th best (j = ceil(k / shards)):
 *                 ONE element-wise MAX all-reduce of the slice [b] over the shards combines both.  The second bound is
 *                 only valid AFTER that reduction over all `shards` shards (with a single shard pass j = k);
 *   finish_batch  applies max([b][0], -[b][1]) and writes rows [b*batch_rows, ...) of this shard's (D, I);
 *   end           after every batch has finished (stream-ordered): repairs overflowed queries, closes the search. */
int knn_index_search_begin_dev(knn_index* idx, int64_t nq, const float* xq_dev, int64_t k, int64_t* nbatches_out,
                               int64_t* batch_rows_out, void* stream);
/* begin for queries of element type `dtype` (KNN_DTYPE_*); the batch calls below read them in that type. */
int knn_index_search_begin_typed_dev(knn_index* idx, int64_t nq, const void* xq_dev, int dtype, int64_t k,
                                     int64_t* nbatches_out, int64_t* batch_rows_out, void* stream);
int knn_index_search_filter_batch_dev(knn_index* idx, int64_t b, int64_t j, float* bounds_dev, void* stream);
int knn_index_search_finish_batch_dev(knn_index* idx, int64_t b, const float* bounds_dev, float* D_dev, int64_t* I_dev,
                                      int64_t id_base, void* stream);
int knn_index_search_end_dev(knn_index* idx, float* D_dev, int64_t* I_dev, int64_t id_base, void* stream);

/* Filtered search (faiss SearchParameters / IDSelector on IndexFlat): restrict a search to selected rows and exclude one
 * row per query, inside the kernels.
 * Contract: a filtered search returns exactly what the unfiltered search returns on an index that holds only the
 * eligible rows, with ids mapped back to the original row numbers - the same D and I bits (the exact rescoring of a
 * (query, row) pair does not depend on the other rows, and the mapping preserves the lower-id-first tie rule).
 *   Row selector (shared by every query of the call): row r is eligible iff allow_bit0 + r < allow_nbits and bit
 *     allow_bit0 + r of allow_bits is set.  allow_bits is an array of 32-bit words, least significant bit first: its
 *     byte layout is faiss's IDSelectorBitmap (bit i & 7 of byte i >> 3).  Bits past allow_nbits select nothing;
 *     allow_bit0 lets one global bitmap serve every shard of a row-sharded database.  NULL: every row is eligible.
 *   Per-query exclusion: exclude_ids[q] is one id in the space the call returns (row + id_base); that row is never
 *     returned for query q.  -1, or an id outside the index, excludes nothing.  NULL: no exclusions.
 * When fewer than k rows remain for a query the tail is padded as for k > ntotal (id -1, -FLT_MAX / +FLT_MAX).  The
 * statistics keep their meaning.  p == NULL is the unfiltered call.  Negative allow_bit0, allow_nbits or id_base, and
 * filter arrays in the wrong memory space (device calls: device memory of the index's device; host calls: not device
 * memory), return KNN_ERR_INVALID.  The host form copies the bitmap words that cover the index and the nq ids to the
 * device; the device forms read the caller's arrays, which must stay valid until the search is done (for
 * begin_params: until search_end). */
typedef struct knn_search_params {
    const uint32_t* allow_bits; int64_t allow_bit0; int64_t allow_nbits; /* NULL: every row */
    const int64_t* exclude_ids;                                          /* NULL: none; nq ids, -1 = none */
} knn_search_params;
/* index.search(xq, k, params=SearchParameters(sel=...)) on host arrays (ids are row numbers). */
int knn_index_search_params(knn_index* idx, int64_t nq, const void* xq, int dtype, int64_t k, float* D, int64_t* I,
                            const knn_search_params* p);
int knn_index_search_params_dev(knn_index* idx, int64_t nq, const void* xq_dev, int dtype, int64_t k, float* D_dev,
                                int64_t* I_dev, int64_t id_base, const knn_search_params* p, void* stream);
/* knn_index_search_begin_typed_dev with a filter; the filter_batch, finish_batch and end calls that follow apply it, and
 * finish_batch and end must be given this id_base (otherwise KNN_ERR_INVALID).  The one-shot search_filter_dev /
 * search_finish_dev pair has no filtered form. */
int knn_index_search_begin_params_dev(knn_index* idx, int64_t nq, const void* xq_dev, int dtype, int64_t k, int64_t id_base,
                                      const knn_search_params* p, int64_t* nbatches_out, int64_t* batch_rows_out,
                                      void* stream);

/* Copy rows [i0, i0+n) back to the host as float32 (faiss Index::reconstruct_n); feeds
 * write_index (pfam/proteins_search.py:39-40). */
int knn_index_reconstruct(knn_index* idx, int64_t i0, int64_t n, float* out);

/* Cross-shard merge (new; the reference is single-process): `nlists` sorted (D, I) results of
 * shape (nq,k), laid out [list][nq][k] in device memory (e.g. the output of an NCCL
 * all-gather), are merged per query into the best k, same ordering rules as search. */
int knn_merge_topk_dev(int metric, int64_t nq, int64_t k, int nlists, const float* D_lists_dev,
                       const int64_t* I_lists_dev, float* D_out_dev, int64_t* I_out_dev, void* stream);

/* Cross-shard exchange fused with the merge, over NVLink peer memory (new; DESIGN.md section 6).  One process
 * per GPU: every rank allocates an exchange buffer (plain cudaMalloc, so it can be exported), publishes its
 * 64-byte CUDA IPC handle to the other ranks (any transport: a host collective, a file, MPI) and maps theirs.
 * knn_merge_topk_peer_dev then merges queries [q0, q1) - this rank's slice - reading rank l's sorted per-shard
 * (D, I) rows through D_peer[l] / I_peer[l] (layout [nq][k], global ids) and storing the merged rows into every
 * rank's D_out_peer[l] / I_out_peer[l].  The pointer arrays are HOST arrays of `nranks` device pointers valid on
 * the calling device (own buffer or mapped peers).  The caller orders it between two barriers: all per-shard
 * results written before, all ranks' merge kernels finished before anyone reads its output. */
int knn_peer_buffer_alloc(void** dev_ptr_out, int64_t bytes, int device);
int knn_peer_buffer_free(void* dev_ptr);
int knn_peer_handle_get(const void* dev_ptr, unsigned char* handle64);
int knn_peer_handle_open(const unsigned char* handle64, int device, void** dev_ptr_out);
int knn_peer_handle_close(void* dev_ptr);
int knn_merge_topk_peer_dev(int metric, int64_t nq, int64_t k, int nranks, int64_t q0, int64_t q1,
                            const void* const* D_peer, const void* const* I_peer, void* const* D_out_peer,
                            void* const* I_out_peer, void* stream);

/* Bound exchange of the two-phase search over the same peer memory, so that it can run per query batch on a side
 * stream next to the GEMM of the following batch (an NCCL kernel does not fit next to a resident GEMM CTA).
 * push:     stores src_dev[0..n) into slot [rank] of EVERY rank's slot array (slots_peer[l] = address of rank l's
 *           float array [nranks][n] as mapped on this device) and then raises flags_peer[l][rank] to `epoch`
 *           (release, system scope).  counter_dev: one zero-initialised uint32 of scratch on this device.
 * wait_max: waits until all `nranks` local flags have reached `epoch` (acquire, system scope; gives up after ~4 s and
 *           sets *timeout_flag_dev instead of hanging), then out_dev[i] = max over ranks of slots_dev[r][i].
 * Epochs increase from call to call; the caller separates two uses of the same slots by a barrier (the result merge). */
int knn_bounds_push_peer_dev(int nranks, int rank, int64_t n, const float* src_dev, void* const* slots_peer,
                             void* const* flags_peer, uint32_t epoch, uint32_t* counter_dev, void* stream);
int knn_bounds_wait_max_dev(int nranks, int64_t n, const float* slots_dev, const uint32_t* flags_dev, uint32_t epoch,
                            float* out_dev, int* timeout_flag_dev, void* stream);

/* ---- Downstream of search: what the reference does with (D, I) next (SURVEY.md section 8, rows f3/f4). ----
 * All pointers are device pointers; I is the (nq,k) int64 matrix index.search returned, D its float32 scores.
 * Label gathers keep Python/numpy index semantics: a negative id counts from the end (id -1 -> last row).
 * `err_dev` is a caller-zeroed int the kernels OR flags into: 1 = NaN score where the reference raises
 * ValueError, 2 = id out of range (IndexError), 4 = infinite score with clip = 0 (OverflowError). */

/* seqvec_search/main.py:53-82 (evaluate_faiss + evaluate): lead[q] = length of the leading run of hits whose
 * family equals the query's (AUC1 numerator), tp[q] = number of such hits (TP numerator).  The common
 * denominator, the family's size in the database (main.py:68), is a bincount the caller does once. */
int knn_eval_family_dev(int64_t nq, int64_t k, const int64_t* I_dev, const int32_t* query_family_dev,
                        const int32_t* db_family_dev, int64_t n_db, int32_t* lead_dev, int32_t* tp_dev, int* err_dev,
                        void* stream);

/* cath/cath.py:76-84 (compute_is_correct), all-vs-all: out[q][l][h] = mapping[q][l] == mapping[I[q][h]][l],
 * mapping = (n_db, levels) int32 label codes, out = (nq, levels, k) bytes. */
int knn_eval_levels_dev(int64_t nq, int64_t k, const int64_t* I_dev, const int32_t* mapping_dev, int levels, int64_t n_db,
                        uint8_t* out_dev, int* err_dev, void* stream);

/* pfam/proteins.py:201-207 (compute_correctness_array) and pfam/proteins_shared.py:139-157 (compute_auc1):
 * per-query sets of homologous database rows in CSR form (set_offsets (nq+1), members sorted ascending within a
 * set).  correct[q][h] = I[q][h] in set q (plain value membership); lead[q] = leading run of member hits, ids
 * wrapped by n_db_wrap first when it is > 0 (target_ids[hit]).  Either output may be NULL. */
int knn_eval_sets_dev(int64_t nq, int64_t k, const int64_t* I_dev, const int64_t* set_offsets_dev,
                      const int64_t* set_members_dev, int64_t n_db_wrap, uint8_t* correct_dev, int32_t* lead_dev,
                      void* stream);

/* pfam/proteins.py:85-122 (remove_self_hit), in place: the first occurrence of self_ids[q] (q itself when
 * self_ids_dev is NULL) in row q - or the last column when it is absent, counted in *n_missing_dev - is rotated
 * to column 0; the caller then drops column 0 (cath/search.py:26 drops it blindly).  D_dev may be NULL. */
int knn_remove_self_hit_dev(int64_t nq, int64_t k, int64_t* I_dev, float* D_dev, const int64_t* self_ids_dev,
                            uint64_t* n_missing_dev, void* stream);

/* seqvec_search/mmseqs/_write_prefilter_db.py:52-97 (write_prefilter_db): the text of the MMseqs2 prefilter
 * database.  Data file: per query, one line "<train_map[hit]>\t<int(clip(score,-1e30,1e30)*100)>\t0\n" per hit
 * != -1 (float32 arithmetic, truncation toward zero, exact for every finite value), then a NUL.  Index file: per
 * query "<test_map[queries[q]]>\t<offset>\t<length>\n" (queries_dev NULL = 0..nq-1).
 * measure: sec_off_dev[0..nq] = byte offset of every query's section (sec_off[nq] = data file size),
 *          idx_off_dev[0..nq] likewise for the index lines.
 * emit:    writes both texts into caller buffers of those sizes (data_dev 16-byte aligned). */
int knn_prefilter_measure_dev(int64_t nq, int64_t k, const int64_t* I_dev, const float* D_dev, const int64_t* queries_dev,
                              const int64_t* test_map_dev, int64_t n_test, const int64_t* train_map_dev, int64_t n_train,
                              int clip, int64_t* sec_off_dev, int64_t* idx_off_dev, int* err_dev, void* stream);
int knn_prefilter_emit_dev(int64_t nq, int64_t k, const int64_t* I_dev, const float* D_dev, const int64_t* queries_dev,
                           const int64_t* test_map_dev, int64_t n_test, const int64_t* train_map_dev, int64_t n_train,
                           int clip, const int64_t* sec_off_dev, const int64_t* idx_off_dev, uint8_t* data_dev,
                           uint8_t* index_dev, int* err_dev, void* stream);

/* Tuning / introspection.  Parameters: "path" (0 auto, 1 exact fp32 scan, 2 tensor-core
 * filter + rerank), "query_batch", "profile" (1: time the dominant kernel with CUDA events),
 * "cta_group" (tcgen05 cta_group of the GEMM kernel, 1 or 2), "tensor_min_nq", "tensor_min_n",
 * "shadow_fmt" (16-bit format of the tensor-core operands: 0 automatic - fp16 where the exact rescoring
 * dominates and the data fits its range, bf16 where the GEMM does -, 1 bf16, 2 fp16; results never depend on it),
 * "mantissa_bits" (experiments: mantissa bits kept in bf16 operands, 0 = all 7), "stream_kernel" (1: launches
 * with <= 64 queries use the few-queries variant of the GEMM kernel; default on), "gemm_stages", "panel_ratio".
 * Statistics of the last search: "path", "launches", "gemm_launches", "gemm_ms", "rerank_ms", "overflow_batches",
 * "overflow_queries"; of the index: "capacity", "shadow_fmt" (1 bf16, 2 fp16), "mantissa_bits",
 * "shadow_conversions" (times the shadow rows were rewritten in the other format).
 * "overlap_finish" (default 1): a search of several query batches runs the exact rescoring of batch b on an internal
 * side stream under the tensor-core filter of batch b + 1; "split_single_batch" (default 1): a one-batch call with
 * k >= 256 is cut into up to four batches for the same reason; "stream_pair" (default 1): 65..128 queries on the
 * CTA-pair form of the few-queries kernel.  Measured-and-rejected variants kept as opt-ins (never change results):
 * "l2_blocked_rerank", "stream_quad", "small_m128". */
int knn_index_set_param(knn_index* idx, const char* name, int64_t value);
int knn_index_get_stat(const knn_index* idx, const char* name, double* out);

/* Total number of kernels this library has launched in this process. */
int64_t knn_kernel_launches(void);

#ifdef __cplusplus
}
#endif
#endif /* KNN_B200_H */

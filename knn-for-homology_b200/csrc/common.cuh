// Shared declarations for libknn_b200.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdint>
#include <cstdio>

#include "../../include/knn_b200.h"

namespace knn {

// ---- error plumbing -------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define KNN_CHECK_CUDA(expr)                                                              \
    do {                                                                                  \
        cudaError_t e__ = (expr);                                                         \
        if (e__ != cudaSuccess) {                                                         \
            knn::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, \
                           __LINE__);                                                     \
            return e__ == cudaErrorMemoryAllocation ? KNN_ERR_MEMORY : KNN_ERR_CUDA;      \
        }                                                                                 \
    } while (0)

#define KNN_CHECK(expr)            \
    do {                           \
        int rc__ = (expr);         \
        if (rc__ != KNN_OK) return rc__; \
    } while (0)

#define KNN_CHECK_LAUNCH()                        \
    do {                                          \
        knn::count_launch();                      \
        KNN_CHECK_CUDA(cudaGetLastError());       \
    } while (0)

// ---- device selection -----------------------------------------------------------------
// Entry points never rely on the caller's current device: knn_index_* calls select the index's device, the
// stateless *_dev calls select the device that owns the memory they are handed (PtrDeviceGuard).
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    DeviceGuard() {}
    explicit DeviceGuard(int dev) { select(dev); }
    void select(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; prev = -1; }
        if (ok && dev >= 0 && prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};
// device ordinal that owns a device allocation (-1: not a device pointer / unknown: the current device stays)
inline int device_of_pointer(const void* p) {
    if (!p) return -1;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) ? a.device : -1;
}
struct PtrDeviceGuard : DeviceGuard {
    explicit PtrDeviceGuard(const void* p) { select(device_of_pointer(p)); }
};
int num_sms();  // SM count of the CURRENT device (cached per device)

// ---- layout constants -----------------------------------------------------------------
constexpr int kDimAlign = 64;        // rows are padded with zeros to a multiple of 64 elements
constexpr uint32_t kInvalidId = 0xFFFFFFFFu;
constexpr int kSortCap = 4096;       // elements sorted in shared memory by one CTA
constexpr int kSelectThreads = 512;

inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// ---- ordering keys --------------------------------------------------------------------
// 64-bit composite key, larger = better:  [ orderable(score) | ~id ].  All valid keys are
// distinct (ids are), so "top-k by key" has no ties and the rule "equal score -> lower id
// first" falls out of the ~id in the low word.  0 is the invalid / padding key (NaN scores
// map to it: like faiss, a NaN never enters a result).
__host__ __device__ inline uint32_t orderable_f32(float f) {
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(f);
#else
    union { float f; uint32_t u; } c; c.f = f; uint32_t u = c.u;
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ inline float from_orderable_f32(uint32_t u) {
    u = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}
// `largest`: 1 when a larger score is better (IP), 0 when a smaller one is (L2 distance).
__host__ __device__ inline uint64_t make_key(float score, uint32_t id, int largest) {
    if (score != score || id == kInvalidId) return 0ull;
    uint32_t o = orderable_f32(score);
    if (!largest) o = ~o;
    return (uint64_t(o) << 32) | uint64_t(~id);
}
__host__ __device__ inline float key_score(uint64_t key, int largest) {
    uint32_t o = uint32_t(key >> 32);
    if (!largest) o = ~o;
    return from_orderable_f32(o);
}
__host__ __device__ inline uint32_t key_id(uint64_t key) { return ~uint32_t(key); }

// ---- kernel launchers (one translation unit each) ---------------------------------------
struct DbStats {          // device-resident, updated by the ingest kernel with atomicMax on
    unsigned max_norm2;   // float bits (values are >= 0, so the uint order is the float order)
    unsigned max_dnorm2;  // max |y - shadow(y)|^2
};

// 16-bit format of the tensor-core operands (the "shadow" copies of database rows and queries).  Both feed
// tcgen05.mma kind::f16 at the same rate; fp16 carries 3 more mantissa bits, i.e. an 8 x smaller rounding term
// in the error bound, but a narrow exponent range - out-of-range values saturate / flush to zero at conversion
// and show up in the MEASURED |y - shadow(y)|, so the bound stays rigorous for either format.
enum ShadowFmt : int { kFmtBF16 = 0, kFmtFP16 = 1 };
typedef uint16_t h16_t;   // raw 16-bit storage of a shadow element

// kernels_basic.cu
int launch_normalize_l2(float* x, int64_t n, int64_t d, cudaStream_t s);
// Element size of a caller row element of dtype KNN_DTYPE_* (0: unknown dtype).
inline size_t dtype_size(int dtype) {
    return dtype == KNN_DTYPE_F32 ? 4 : (dtype == KNN_DTYPE_F16 || dtype == KNN_DTYPE_BF16) ? 2 : 0;
}

// src rows of d elements of `src_dtype` (KNN_DTYPE_*, stride src_ld elements) -> zero-padded fp32 master rows
// (optional), 16-bit shadow rows in format `fmt`, |y|^2 (optional) and the running maxima in *stats.  16-bit source
// rows are converted exactly to fp32 at the load: every output equals that of the up-converted rows, bit for bit.
// shadow_is_master: the rounded values ARE the row.
// mbits: explicit mantissa bits kept in a bf16 shadow (7 = all of them; ignored for fp16 and for master rows).
int launch_ingest(const void* src, int src_dtype, int64_t src_ld, int64_t n, int d, int dp, float* dst_f32, h16_t* dst_h16,
                  int fmt, int mbits, bool shadow_is_master, float* norms2, DbStats* stats, cudaStream_t s);
// Queries (rows of d elements of `xq_dtype`) -> zero-padded fp32 (ld = dp) and 16-bit copies, |x|^2 and the score
// error bound eps (see DESIGN.md "error bound"); rows [nq, nq_pad) of the 16-bit copy are zeroed.
int launch_prep_queries(const void* xq, int xq_dtype, int64_t nq, int64_t nq_pad, int d, int dp, float* xq_f32,
                        h16_t* xq_h16, int fmt, int mbits, float* xnorm2, float* eps, const DbStats* stats,
                        int metric, cudaStream_t s);
// Exact fp32 scores of queries [0, nqt) (nqt <= kScanMaxQueries... looped inside) against rows
// [j0, j1): out[q * ld_out + (j - j0)] = <x_q, y_j> (IP) or max(0, |x|^2 + |y|^2 - 2<x,y>) (L2).
int launch_scan_f32(const float* xq_f32, const float* xnorm2, int64_t nq, int dp, const float* xb_f32,
                    const __nv_bfloat16* xb_bf16, const float* ynorm2, int64_t j0, int64_t j1, int metric,
                    float* out, int64_t ld_out, cudaStream_t s);
// Exact rescoring of candidate lists in place: for every query q and slot i < min(count[q], cap)
// with approx score >= tau[q], scores[q*cap+i] <- exact fp32 score (same arithmetic as the scan
// kernel); other slots get id = kInvalidId.
int launch_rerank(const float* xq_f32, const float* xnorm2, int64_t nq, int dp, const float* xb_f32,
                  const __nv_bfloat16* xb_bf16, const float* ynorm2, int metric, float* cand_scores,
                  uint32_t* cand_ids, const int* counts, const float* tau, int cap, int64_t ntotal, int k, int l2_blocked,
                  cudaStream_t s);

// select.cu
// Level 1: dense rows -> per (query, segment) best-k appended to lists[q][seg*k + r].
int launch_select_dense(const float* scores, int64_t ld, int64_t ncols, int64_t nq, int seg_len,
                        uint32_t id_base, int k, int largest, float* list_scores, uint32_t* list_ids,
                        int64_t list_ld, int64_t list_off, cudaStream_t s);
// Final: lists[q][0..len) (len = counts ? min(counts[q], list_ld) : fixed_len) -> sorted D/I rows.
int launch_select_final(const float* list_scores, const uint32_t* list_ids, const int* counts,
                        int64_t list_ld, int64_t fixed_len, int64_t nq, int k, int largest, float* D,
                        int64_t* I, int64_t id_base, cudaStream_t s);
// Merge of [nlists][nq][k] (float, int64) results.
int launch_merge_lists(const float* D_lists, const int64_t* I_lists, int nlists, int64_t nq, int k,
                       int largest, float* D, int64_t* I, cudaStream_t s);

// gemm_sm100.cu  (tcgen05 / TMEM / TMA)
struct FilterState {        // per query-batch, device resident
    float* thr;             // [nq_pad] running candidate threshold (approx-score domain)
    int* counts;            // [nq_pad] appended candidates (may exceed cap: overflow marker)
    float* cand_scores;     // [nq_pad * cap]
    uint32_t* cand_ids;     // [nq_pad * cap]
    int cap;
    int* ovf;               // [nq] sticky per-query flag: the list ran past its capacity at some panel
};
struct GemmPlan;            // opaque: tensor maps + launch geometry
int gemm_plan_create(GemmPlan** out, int device);
void gemm_plan_destroy(GemmPlan* p);
void gemm_plan_set_cta_group(GemmPlan* p, int cg);          // 1 or 2 (default 2: CTA pairs)
void gemm_plan_set_l2_hints(GemmPlan* p, int on);
void gemm_plan_set_debug(GemmPlan* p, int skip_epilogue);
void gemm_plan_set_stages(GemmPlan* p, int stages);
void gemm_plan_set_stream_kernel(GemmPlan* p, int on);   // few-queries variant for launches with <= 64 queries (default on)
void gemm_plan_set_stream_pair(GemmPlan* p, int on);     // 65..128 queries: CTA-pair form of the few-queries variant (default on)
void gemm_plan_set_stream_quad(GemmPlan* p, int on);     // experiments: 129..256 queries on two pairs per cluster, database tiles multicast (default off)
void gemm_plan_set_small_m128(GemmPlan* p, int on);      // 65..128 queries: single-CTA (M = 128) tiles (default on)
int gemm_plan_query_rows_multiple(const GemmPlan* p);     // nq_pad granularity of the chosen variant
// Scores queries (16-bit, format fmt_q, [nq_pad x dp]) against database rows [j0, j1) (16-bit, format fmt_db,
// [ntotal x dp]) on the tensor cores and appends every (score, id) with score >= thr[q] to the candidate lists.
// dense_first: rows are stored at slot (j - j0) without atomics (first panel, thr = -inf).
int gemm_filter_launch(GemmPlan* p, const h16_t* xq_h16, int fmt_q, int64_t nq, int64_t nq_pad, int dp,
                       const h16_t* xb_h16, int fmt_db, int64_t ntotal, const float* ynorm2, int64_t j0,
                       int64_t j1, int metric, bool dense_first, FilterState st, cudaStream_t s);
// After a panel: thr[q] <- (k-th best approx score so far) - 2*eps[q]; drops candidates below the
// new threshold; raises *overflow when a list ran past its capacity.
int launch_tighten(FilterState st, const float* eps, int64_t nq, int k, int compact, float* tau_out,
                   int* overflow, cudaStream_t s);
// thr <- -FLT_MAX (real queries) / +FLT_MAX (padding rows); counts <- first_count / 0.
int launch_init_filter(FilterState st, int64_t nq, int64_t nq_pad, int first_count, cudaStream_t s);
// Two-phase (sharded) search: lower[q] = thr + eps on the way out; thr <- max(thr, lower - eps) on the way in.
int launch_export_lower(const float* thr, const float* eps, int64_t nq, float* lower, cudaStream_t s);
// lower_j[q] = (j-th best approximate score in the list) - eps[q]
// (negate: the value is written with its sign flipped, so that an element-wise MAX reduction yields the MIN)
int launch_kth_lower(FilterState st, const float* eps, int64_t nq, int j, bool negate, float* lower_j, cudaStream_t s);
// thr <- max(thr, max(lower, -neg_lower2) - eps); neg_lower2 may be null
int launch_apply_lower(float* thr, const float* eps, const float* lower, const float* neg_lower2, int64_t nq, cudaStream_t s);
int launch_fill_f32(float* p, int64_t n, float v, cudaStream_t s);
// Overflow repair: out[i] = float(xq[idx[i]]) (rows of d elements of xq_dtype, written as fp32);
// D[idx[i]] = Dt[i], I[idx[i]] = It[i] (rows of k).
int launch_gather_rows(const void* xq, int xq_dtype, int d, const int* idx, int64_t n, float* out, cudaStream_t s);
int launch_scatter_results(const float* Dt, const int64_t* It, const int* idx, int64_t n, int k, float* D, int64_t* I,
                           cudaStream_t s);

}  // namespace knn

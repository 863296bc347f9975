// C ABI of libknn_b200.so and the host-side orchestration of a search.
//
// Replaces, for the flat path only, the faiss calls of the reference drivers (paths relative
// to /root/reference): faiss.normalize_L2 (cath/search.py:19), faiss.IndexFlat
// (cath/search.py:20), index.add (cath/search.py:22), index.search (cath/search.py:24,
// pfam/proteins_search.py:49, seqvec_search/main.py:45).
//
// Two device paths, both CUDA only:
//   exact  : fp32 scan kernel -> dense scores -> two-level radix select          (small nq / small N)
//   tensor : tcgen05 GEMM over 16-bit shadow copies (fp16 or bf16) with threshold-filter epilogue over growing database panels,
//            per-panel threshold tightening, exact fp32 rerank of the surviving candidates,
//            final radix select                                                   (large batches)
// The tensor path returns exactly what the exact path returns: the filter keeps a provable
// superset of the true top-k (DESIGN.md "error bound") and the rerank recomputes the scores
// with the scan kernel's arithmetic.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"

namespace knn {

static thread_local std::string g_error;
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_error = buf;
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// Large workspaces (candidate lists: ~1 GB per index) outlive the index that allocated them in a small per-device
// pool: the reference's drivers build a NEW index per embedding matrix (cath/search.py:20 inside a loop over ~20
// files and 2 metrics), and a cudaMalloc + cudaFree of a gigabyte per call costs more than the search of a CATH-sized
// matrix (measured: 13 ms vs up to 175 ms per cath.search.search call depending on the box's allocator state).
struct WorkspacePool {
    struct Entry { void* p; size_t bytes; int device; };
    std::mutex mu;
    std::vector<Entry> free_list;
    size_t pooled = 0;
    static constexpr size_t kMinBytes = size_t(32) << 20, kMaxPooled = size_t(6) << 30;
    void* take(size_t want, int device, size_t* got) {
        std::lock_guard<std::mutex> g(mu);
        size_t best = free_list.size();
        for (size_t i = 0; i < free_list.size(); ++i)
            if (free_list[i].device == device && free_list[i].bytes >= want && free_list[i].bytes <= want + want / 2 &&
                (best == free_list.size() || free_list[i].bytes < free_list[best].bytes))
                best = i;
        if (best == free_list.size()) return nullptr;
        Entry e = free_list[best];
        free_list.erase(free_list.begin() + long(best));
        pooled -= e.bytes;
        *got = e.bytes;
        return e.p;
    }
    bool give(void* p, size_t bytes, int device) {
        if (bytes < kMinBytes) return false;
        std::lock_guard<std::mutex> g(mu);
        if (pooled + bytes > kMaxPooled) return false;
        free_list.push_back({p, bytes, device});
        pooled += bytes;
        return true;
    }
};
static WorkspacePool g_pool;
static WorkspacePool g_pinned_pool;  // page-locked bounce buffers (device = -1)

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int ensure(size_t want) {
        if (want <= bytes) return KNN_OK;
        release();
        int dev = 0;
        cudaGetDevice(&dev);
        if (want >= WorkspacePool::kMinBytes) {
            size_t got = 0;
            if (void* q = g_pool.take(want, dev, &got)) {
                p = q;
                bytes = got;
                return KNN_OK;
            }
        }
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_error("cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
            return KNN_ERR_MEMORY;
        }
        bytes = want;
        return KNN_OK;
    }
    // Callers release only when no work that touches the buffer is in flight (index destruction synchronises first;
    // growth happens between searches), so a pooled buffer can be handed to the next owner immediately.
    void release() {
        if (p) {
            int dev = 0;
            cudaGetDevice(&dev);
            if (bytes >= WorkspacePool::kMinBytes) cudaDeviceSynchronize();  // what cudaFree would have implied
            if (!g_pool.give(p, bytes, dev)) cudaFree(p);
        }
        p = nullptr;
        bytes = 0;
    }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

struct PinBuf {  // page-locked host memory (bounce buffers of the host-pointer entry points)
    void* p = nullptr;
    size_t bytes = 0;
    int ensure(size_t want) {
        if (want <= bytes) return KNN_OK;
        release();
        if (want >= WorkspacePool::kMinBytes) {
            size_t got = 0;
            if (void* q = g_pinned_pool.take(want, -1, &got)) {
                p = q;
                bytes = got;
                return KNN_OK;
            }
        }
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        if (e != cudaSuccess) {
            cudaGetLastError();
            p = nullptr;
            set_error("cudaHostAlloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
            return KNN_ERR_MEMORY;
        }
        bytes = want;
        return KNN_OK;
    }
    void release() {
        if (p) {
            if (bytes >= WorkspacePool::kMinBytes) cudaDeviceSynchronize();
            if (!g_pinned_pool.give(p, bytes, -1)) cudaFreeHost(p);
        }
        p = nullptr;
        bytes = 0;
    }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

// Staging copies between pageable caller memory and the pinned bounce buffers run on the calling thread while the
// GPU works; one core moves ~8-10 GB/s, so large blocks are split over a few threads.
inline void host_copy(void* dst, const void* src, size_t bytes) {
    const size_t kMin = size_t(8) << 20;
    unsigned nt = unsigned(std::min<size_t>(4, bytes / kMin));
    if (nt <= 1) {
        memcpy(dst, src, bytes);
        return;
    }
    std::vector<std::thread> th;
    const size_t per = ((bytes / nt) + 4095) & ~size_t(4095);
    for (unsigned t = 1; t < nt; ++t) {
        const size_t off = size_t(t) * per;
        if (off >= bytes) break;
        const size_t len = std::min(per, bytes - off);
        th.emplace_back([=] { memcpy(static_cast<char*>(dst) + off, static_cast<const char*>(src) + off, len); });
    }
    memcpy(dst, src, std::min(per, bytes));
    for (auto& t : th) t.join();
}

// Row `row` of a caller matrix of d elements of dtype KNN_DTYPE_* (queries and added rows may be fp32, fp16 or bf16).
inline const void* row_at(const void* base, int64_t row, int d, int dtype) {
    return static_cast<const char*>(base) + size_t(row) * size_t(d) * dtype_size(dtype);
}

inline int check_dtype(int dtype, const char* who) {
    if (dtype_size(dtype) == 0) {
        set_error("%s: unknown dtype %d (KNN_DTYPE_F32, KNN_DTYPE_F16 or KNN_DTYPE_BF16)", who, dtype);
        return KNN_ERR_INVALID;
    }
    return KNN_OK;
}

// true when the driver can DMA straight to / from p (cudaHostAlloc / cudaHostRegister memory)
inline bool host_pointer_is_pinned(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

}  // namespace knn

using namespace knn;

struct knn_index {
    int d = 0, dp = 0, metric = 0, device = 0;
    unsigned flags = 0;
    int64_t ntotal = 0, capacity = 0;
    float* xb_f32 = nullptr;          // [capacity x dp] zero-padded rows (absent with BF16_STORAGE)
    h16_t* xb_h16 = nullptr;          // [capacity x dp] 16-bit shadow rows, format shadow_fmt (bf16 with BF16_STORAGE: the rows themselves)
    int shadow_fmt = kFmtBF16;        // format of ALL shadow rows (see desired_shadow / prepare_shadow)
    int shadow_mbits = 7;             // explicit mantissa bits kept in bf16 shadow rows
    bool stats_dirty = false;         // rows were added since the shadow's rounding error was last looked at
    bool fp16_unfit = false;          // the data leaves fp16's exponent range (measured): automatic choice stays bf16
    float* ynorm2 = nullptr;          // [capacity]
    DbStats* stats = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t add_event = nullptr;  // last ingest; searches on another stream wait on it
    cudaEvent_t search_event = nullptr;  // end of the last search (it may rewrite the shadow rows / stats): adds and resets wait on it
    GemmPlan* plan = nullptr;
    // workspaces: exact path / staging
    DevBuf stage, xq_f32, xnorm2, eps, scores, lists_s, lists_i, overflow;
    DevBuf ovf_q, ovf_idx, ovf_x, ovf_D, ovf_I;  // per-query overflow flags of a call and the repair staging
    DevBuf h_xq, h_D, h_I;
    // host-pointer search, pipelined per query batch (HostPipe below): two slots of device staging, pinned bounce
    // buffers for pageable caller memory, one copy stream per direction
    DevBuf hp_xq[2], hp_D[2], hp_I[2];
    PinBuf hp_pin_xq[2], hp_pin_D[2], hp_pin_I[2];
    DevBuf stage2;                      // second ingest staging buffer (knn_index_add double-buffers the H2D copies)
    cudaStream_t copy_in = nullptr, copy_out = nullptr;
    cudaEvent_t hp_in_ready[2] = {nullptr, nullptr}, hp_out_done[2] = {nullptr, nullptr}, hp_computed[2] = {nullptr, nullptr};
    cudaEvent_t hp_in_free[2] = {nullptr, nullptr};
    cudaEvent_t stage_free[2] = {nullptr, nullptr};
    // tensor path: per-query state of the filter (queries, thresholds, candidate lists)
    struct TensorWs {
        DevBuf xq_f32, xq_h16, xnorm2, eps, thr, counts, cand_s, cand_i;
    };
    TensorWs ws1[2];  // one query batch each (single-call search): batch b filters in ws1[b & 1] while batch b - 1 finishes
    TensorWs ws2;     // all queries of a two-phase search (filter ... exchange ... finish)
    cudaStream_t side = nullptr;                  // finish phase of batch b runs here, under the GEMM of batch b + 1 (lowest priority)
    cudaStream_t hi = nullptr;                    // filter phase of an overlapped search (highest priority, see search_tensor)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaEvent_t ev_filtered[2] = {nullptr, nullptr};  // filter of the batch in ws1[i] done (main stream)
    cudaEvent_t ev_finished[2] = {nullptr, nullptr};  // finish of the batch in ws1[i] done (side stream): ws1[i] reusable
    int overlap_finish = 1;
    int split_single_batch = 1;
    struct Pending {
        bool active = false, tensor = false;
        int64_t nq = 0, qb = 0, nbatches = 0;
        int k = 0, cap = 0;
        const void* xq = nullptr;    // the caller's queries (kept alive by the caller until search_end) ...
        int dtype = KNN_DTYPE_F32;   // ... and their element type
        long long launches0 = 0;
    } pend;
    // parameters
    int path_param = 0;
    int64_t query_batch = 16384;
    int profile = 0;
    int64_t tensor_min_nq = 1, tensor_min_n = 8192;  // measured: the bf16 stream beats the fp32 scan from nq = 1 (profiles/)
    int cta_group = 2;
    int l2_hints = 0;
    int debug_skip_epilogue = 0;
    int gemm_stages = 0;
    int stream_kernel = 1;
    int stream_pair = 1;
    int dense_small_db = 1;
    int stream_quad = 0;  // measured: 7.4 ms against the main kernel's 6.0 ms at 256 queries x 10M rows (gemm_sm100.cu)
    int l2_blocked_rerank = 0;  // opt-in: cuts the rerank's DRAM bytes 10 x but is 2 x slower (see kernels_basic.cu)
    int small_m128 = 0;  // measured slower than the CTA-pair tiles (5.9 vs 4.6 ms at 128 queries x 10M rows): off
    int panel_ratio = 0;  // 0: automatic
    int64_t small_batch_nq = 256;  // batches up to this size use growth ratio 8
    int shadow_param = 0;          // 16-bit format of the tensor-core operands: 0 automatic (desired_shadow), 1 bf16, 2 fp16
    int mbits_param = 0;           // mantissa bits kept in bf16 operands: 0 automatic, 2..7
    // statistics of the last search
    int last_path = 0;
    long long st_launches = 0, st_gemm_launches = 0, st_candidates = 0, st_overflow_batches = 0, st_overflow_queries = 0, st_rerank_pairs = 0, st_shadow_conversions = 0;
    double st_gemm_ms = 0, st_rerank_ms = 0;
    std::vector<cudaEvent_t> ev_pool;   // profile = 1: pairs of events around the GEMM launches ...
    size_t ev_used = 0;
    std::vector<cudaEvent_t> ev_pool_r; // ... and around the rerank launches
    size_t ev_used_r = 0;
};

namespace {

// profile = 1: after the stream has been synchronised, fold the event pairs into the statistics
void collect_profile(knn_index* ix) {
    for (size_t i = 0; i + 1 < ix->ev_used; i += 2) {
        float ms = 0;
        cudaEventElapsedTime(&ms, ix->ev_pool[i], ix->ev_pool[i + 1]);
        ix->st_gemm_ms += ms;
    }
    for (size_t i = 0; i + 1 < ix->ev_used_r; i += 2) {
        float ms = 0;
        cudaEventElapsedTime(&ms, ix->ev_pool_r[i], ix->ev_pool_r[i + 1]);
        ix->st_rerank_ms += ms;
    }
}

constexpr int64_t kMaxRows = 0x7FFFFFFFll;

bool bf16_only(const knn_index* ix) { return (ix->flags & KNN_FLAG_BF16_STORAGE) != 0; }

int grow(knn_index* ix, int64_t want_rows, bool exact = false) {
    if (want_rows <= ix->capacity) return KNN_OK;
    if (want_rows > kMaxRows) {  // TMA row coordinates are signed 32-bit (gemm_sm100.cu); ids are stored as uint32
        set_error("an index (one shard) holds at most 2^31-1 rows");
        return KNN_ERR_LIMIT;
    }
    int64_t cap = exact ? want_rows : ix->capacity + ix->capacity / 2;
    if (cap < want_rows) cap = want_rows;
    if (cap < 1024) cap = 1024;
    if (cap > kMaxRows) cap = kMaxRows;
    // rows may have been ingested on a caller's stream: settle everything before moving them
    KNN_CHECK_CUDA(cudaDeviceSynchronize());
    float* nf = nullptr;
    h16_t* nb = nullptr;
    float* nn = nullptr;
    cudaError_t e = cudaSuccess;
    if (!bf16_only(ix)) e = cudaMalloc(&nf, size_t(cap) * ix->dp * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&nb, size_t(cap) * ix->dp * sizeof(h16_t));
    if (e == cudaSuccess) e = cudaMalloc(&nn, size_t(cap) * sizeof(float));
    if (e != cudaSuccess) {
        cudaGetLastError();
        if (nf) cudaFree(nf);
        if (nb) cudaFree(nb);
        if (nn) cudaFree(nn);
        set_error("cannot allocate storage for %lld rows of %d floats: %s", (long long)cap, ix->dp,
                  cudaGetErrorString(e));
        return KNN_ERR_MEMORY;
    }
    if (ix->ntotal > 0) {
        if (nf) KNN_CHECK_CUDA(cudaMemcpyAsync(nf, ix->xb_f32, size_t(ix->ntotal) * ix->dp * sizeof(float), cudaMemcpyDeviceToDevice, ix->stream));
        KNN_CHECK_CUDA(cudaMemcpyAsync(nb, ix->xb_h16, size_t(ix->ntotal) * ix->dp * sizeof(h16_t), cudaMemcpyDeviceToDevice, ix->stream));
        KNN_CHECK_CUDA(cudaMemcpyAsync(nn, ix->ynorm2, size_t(ix->ntotal) * sizeof(float), cudaMemcpyDeviceToDevice, ix->stream));
        KNN_CHECK_CUDA(cudaStreamSynchronize(ix->stream));
    }
    if (ix->xb_f32) cudaFree(ix->xb_f32);
    if (ix->xb_h16) cudaFree(ix->xb_h16);
    if (ix->ynorm2) cudaFree(ix->ynorm2);
    ix->xb_f32 = nf;
    ix->xb_h16 = nb;
    ix->ynorm2 = nn;
    ix->capacity = cap;
    return KNN_OK;
}

cudaEvent_t next_event_r(knn_index* ix) {
    if (ix->ev_used_r == ix->ev_pool_r.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        ix->ev_pool_r.push_back(e);
    }
    return ix->ev_pool_r[ix->ev_used_r++];
}

cudaEvent_t next_event(knn_index* ix) {
    if (ix->ev_used == ix->ev_pool.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        ix->ev_pool.push_back(e);
    }
    return ix->ev_pool[ix->ev_used++];
}

// ---- 16-bit shadow format -------------------------------------------------------------------
const __nv_bfloat16* bf16_rows(const knn_index* ix) { return reinterpret_cast<const __nv_bfloat16*>(ix->xb_h16); }

constexpr int kAutoMantissaBits = 7;

struct ShadowChoice {
    int fmt, mbits;
};

// Which 16-bit format serves a search of the k best among n rows (k = 0: not known yet, at add time).
// Both formats run tcgen05.mma kind::f16 at the same rate per clock; they differ in two measured ways
// (profiles/r01_shadow_formats.md): fp16's 3 extra mantissa bits shrink the rounding term of the error bound 8 x,
// i.e. fewer candidates to rescore exactly - and they cost multiplier power, which under the board's power cap is
// ~6 % of the clock in a long GEMM.  So fp16 where the rescoring dominates (k large against n), bf16 where the
// GEMM does.  The shadow is rewritten from the fp32 master rows when the regime changes (one pass over the rows).
ShadowChoice desired_shadow(const knn_index* ix, int64_t k, int64_t n) {
    const int mb = ix->mbits_param ? ix->mbits_param : kAutoMantissaBits;
    if (bf16_only(ix)) return {kFmtBF16, 7};  // the bf16 values are the database
    if (ix->shadow_param == 1) return {kFmtBF16, mb};
    if (ix->shadow_param == 2) return {kFmtFP16, 10};
    const bool rescoring_heavy = k > 0 ? n < 10000 * k : n < (int64_t(1) << 20);
    if (rescoring_heavy && !ix->fp16_unfit) return {kFmtFP16, 10};
    return {kFmtBF16, mb};
}

int query_mbits(const knn_index* ix) {
    if (ix->shadow_fmt != kFmtBF16) return 10;
    return bf16_only(ix) ? (ix->mbits_param ? ix->mbits_param : kAutoMantissaBits) : ix->shadow_mbits;
}

// Rewrites every shadow row from the fp32 master rows (and re-measures the rounding error).
int convert_shadow(knn_index* ix, ShadowChoice c, cudaStream_t s) {
    if (ix->ntotal > 0) {
        KNN_CHECK_CUDA(cudaMemsetAsync(ix->stats, 0, sizeof(DbStats), s));
        KNN_CHECK(launch_ingest(ix->xb_f32, KNN_DTYPE_F32, ix->dp, ix->ntotal, ix->dp, ix->dp, nullptr, ix->xb_h16, c.fmt,
                                c.mbits, false, nullptr, ix->stats, s));
        ix->st_shadow_conversions++;
    }
    ix->shadow_fmt = c.fmt;
    ix->shadow_mbits = c.mbits;
    return KNN_OK;
}

// Before a tensor-path search for the k best: bring the shadow rows into the format that serves it.  fp16 is only
// usable while the data sits inside its exponent range: after rows were added (or rewritten) the MEASURED rounding
// error is compared with what bf16 guarantees (|y - bf16(y)| <= 2^-9 |y|); when fp16 does worse than a quarter of
// that on the worst row (saturated or flushed values), the automatic choice falls back to bf16 for this database.
int prepare_shadow(knn_index* ix, int64_t k, cudaStream_t s) {
    if (bf16_only(ix) || ix->ntotal == 0) return KNN_OK;
    ShadowChoice want = desired_shadow(ix, k, ix->ntotal);
    if (want.fmt != ix->shadow_fmt || want.mbits != ix->shadow_mbits) {
        KNN_CHECK(convert_shadow(ix, want, s));
        ix->stats_dirty = true;
    }
    if (ix->stats_dirty && ix->shadow_fmt == kFmtFP16 && ix->shadow_param == 0) {
        DbStats h;
        KNN_CHECK_CUDA(cudaMemcpyAsync(&h, ix->stats, sizeof(h), cudaMemcpyDeviceToHost, s));
        KNN_CHECK_CUDA(cudaStreamSynchronize(s));
        float n2, d2;
        memcpy(&n2, &h.max_norm2, 4);
        memcpy(&d2, &h.max_dnorm2, 4);
        if (d2 > n2 * 9.5367431640625e-07f /* 2^-20 */) {
            ix->fp16_unfit = true;
            KNN_CHECK(convert_shadow(ix, desired_shadow(ix, k, ix->ntotal), s));
        }
    }
    ix->stats_dirty = false;
    return KNN_OK;
}

// ---- exact path ---------------------------------------------------------------------------
int search_exact(knn_index* ix, int64_t nq, const void* xq_dev, int qdt, int k, float* D, int64_t* I, int64_t id_base,
                 cudaStream_t s) {
    const int largest = ix->metric == KNN_METRIC_INNER_PRODUCT;
    const int64_t N = ix->ntotal;
    const int seg_len = 32768;
    const int64_t nseg = (N + seg_len - 1) / seg_len;
    const int64_t list_ld = nseg * k;
    // batch sizes from fixed budgets: lists <= 1 GiB, dense scores <= 512 MiB
    int64_t qb = nq < 1024 ? nq : 1024;
    while (qb > 8 && qb * list_ld * 8 > (int64_t(1) << 30)) qb /= 2;
    int64_t chunk = ((int64_t(512) << 20) / (qb * 4)) / seg_len * seg_len;
    if (chunk < seg_len) chunk = seg_len;
    if (chunk > nseg * seg_len) chunk = nseg * seg_len;
    KNN_CHECK(ix->xq_f32.ensure(size_t(qb) * ix->dp * sizeof(float)));
    KNN_CHECK(ix->xnorm2.ensure(size_t(qb) * sizeof(float)));
    KNN_CHECK(ix->eps.ensure(size_t(qb) * sizeof(float)));
    KNN_CHECK(ix->scores.ensure(size_t(qb) * chunk * sizeof(float)));
    KNN_CHECK(ix->lists_s.ensure(size_t(qb) * list_ld * sizeof(float)));
    KNN_CHECK(ix->lists_i.ensure(size_t(qb) * list_ld * sizeof(uint32_t)));
    for (int64_t q0 = 0; q0 < nq; q0 += qb) {
        const int64_t nb = nq - q0 < qb ? nq - q0 : qb;
        KNN_CHECK(launch_prep_queries(row_at(xq_dev, q0, ix->d, qdt), qdt, nb, nb, ix->d, ix->dp, ix->xq_f32.as<float>(), nullptr,
                                      kFmtBF16, 7, ix->xnorm2.as<float>(), ix->eps.as<float>(), ix->stats, ix->metric, s));
        for (int64_t j0 = 0; j0 < N; j0 += chunk) {
            const int64_t j1 = j0 + chunk < N ? j0 + chunk : N;
            KNN_CHECK(launch_scan_f32(ix->xq_f32.as<float>(), ix->xnorm2.as<float>(), nb, ix->dp, ix->xb_f32,
                                      bf16_rows(ix), ix->ynorm2, j0, j1, ix->metric, ix->scores.as<float>(), chunk, s));
            KNN_CHECK(launch_select_dense(ix->scores.as<float>(), chunk, j1 - j0, nb, seg_len, uint32_t(j0), k, largest,
                                          ix->lists_s.as<float>(), ix->lists_i.as<uint32_t>(), list_ld,
                                          (j0 / seg_len) * k, s));
        }
        KNN_CHECK(launch_select_final(ix->lists_s.as<float>(), ix->lists_i.as<uint32_t>(), nullptr, list_ld, list_ld,
                                      nb, k, largest, D + q0 * k, I + q0 * k, id_base, s));
    }
    return KNN_OK;
}

// ---- tensor path --------------------------------------------------------------------------
// Candidate-list slots per query.  A small database searched for many neighbours (k >= 256 of <= 16,384 rows: C2,
// 14,433 rows, k = 1000) gets one slot per row: with k / N of 7 % a threshold filter lets a quarter of the scores of
// its second panel through - tens of millions of atomic appends - so the whole database is scored as ONE dense panel
// instead (plain coalesced stores), followed by one tighten (measured: C2's GEMM launches 2.9 -> ~0.6 ms).
int candidate_capacity(int k, int64_t ntotal, bool dense_small) {
    int cap = 8192;
    while (cap < 8 * k) cap *= 2;
    if (dense_small && k >= 256 && ntotal > cap && ntotal <= 16384) cap = 16384;
    return cap;
}

int tensor_ws_ensure(knn_index::TensorWs& W, int64_t rows, int dp, int cap) {
    KNN_CHECK(W.xq_f32.ensure(size_t(rows) * dp * sizeof(float)));
    KNN_CHECK(W.xq_h16.ensure(size_t(rows) * dp * sizeof(h16_t)));
    KNN_CHECK(W.xnorm2.ensure(size_t(rows) * sizeof(float)));
    KNN_CHECK(W.eps.ensure(size_t(rows) * sizeof(float)));
    KNN_CHECK(W.thr.ensure(size_t(rows) * sizeof(float)));
    KNN_CHECK(W.counts.ensure(size_t(rows) * sizeof(int)));
    KNN_CHECK(W.cand_s.ensure(size_t(rows) * cap * sizeof(float)));
    KNN_CHECK(W.cand_i.ensure(size_t(rows) * cap * sizeof(uint32_t)));
    return KNN_OK;
}

FilterState filter_state(knn_index::TensorWs& W, int64_t off, int cap, int* ovf = nullptr) {
    FilterState st;
    st.ovf = ovf;
    st.thr = W.thr.as<float>() + off;
    st.counts = W.counts.as<int>() + off;
    st.cand_scores = W.cand_s.as<float>() + off * cap;
    st.cand_ids = W.cand_i.as<uint32_t>() + off * cap;
    st.cap = cap;
    return st;
}

int tensor_prepare(knn_index* ix) {
    if (!ix->plan) KNN_CHECK(gemm_plan_create(&ix->plan, ix->device));
    gemm_plan_set_cta_group(ix->plan, ix->cta_group);
    gemm_plan_set_l2_hints(ix->plan, ix->l2_hints);
    gemm_plan_set_debug(ix->plan, ix->debug_skip_epilogue);
    gemm_plan_set_stages(ix->plan, ix->gemm_stages);
    gemm_plan_set_stream_kernel(ix->plan, ix->stream_kernel);
    gemm_plan_set_small_m128(ix->plan, ix->small_m128);
    gemm_plan_set_stream_pair(ix->plan, ix->stream_pair);
    gemm_plan_set_stream_quad(ix->plan, ix->stream_quad);
    return KNN_OK;
}

// Filter phase of one query batch (rows [off, off+nb) of W): tensor-core scores over database panels of
// growing size, survivors appended to the candidate lists, thresholds tightened after every panel.
// On return thr[q] = (k-th best approximate score) - 2 eps[q].
int tensor_filter_batch(knn_index* ix, knn_index::TensorWs& W, int64_t off, int64_t nb, const void* xq_batch, int qdt, int k,
                        int cap, int* d_overflow, int* d_ovf_q, cudaStream_t s) {
    const int64_t N = ix->ntotal;
    const int64_t nb_pad = round_up(nb, 256);
    // first panel: stored densely (every score), sized so that the list it leaves fits the register-resident
    // tighten (<= 1024 entries) for small k, and holds well over k rows for large k
    int64_t first_panel = std::max<int64_t>(1024, round_up(4 * int64_t(k), 256));
    if (first_panel > cap / 2) first_panel = cap / 2;
    if (first_panel > N) first_panel = N;
    if (ix->dense_small_db && k >= 256 && N <= cap && N <= 16384) first_panel = N;  // one dense panel: no later panel needs room
    // small batches are launch-bound, not list-bound: fewer, faster growing panels (7 k' survivors per panel and query)
    // (only while the ~7 k' survivors of the second panel fit next to the dense first panel: k' ~ 1.7 k)
    const bool fast_growth = nb <= ix->small_batch_nq && 12 * int64_t(k) + first_panel <= cap;
    const int ratio = ix->panel_ratio >= 2 ? ix->panel_ratio : (fast_growth ? 8 : 2);
    FilterState st = filter_state(W, off, cap, d_ovf_q);
    float* xq_f32 = W.xq_f32.as<float>() + off * ix->dp;
    h16_t* xq_h16 = W.xq_h16.as<h16_t>() + off * ix->dp;
    const int fmt_q = ix->shadow_fmt;  // tcgen05.mma kind::f16 takes one 16-bit format per launch (mixing them is an illegal instruction)
    KNN_CHECK(launch_prep_queries(xq_batch, qdt, nb, nb_pad, ix->d, ix->dp, xq_f32, xq_h16, fmt_q, query_mbits(ix),
                                  W.xnorm2.as<float>() + off, W.eps.as<float>() + off, ix->stats, ix->metric, s));
    KNN_CHECK(launch_init_filter(st, nb, nb_pad, int(first_panel), s));
    int64_t j0 = 0;
    int panel = 0;
    while (j0 < N) {
        // rows seen after each panel: P, 4P, 8P, 16P, ... (P = first, densely stored panel).  A panel runs with the
        // threshold of its start, so it appends about (r - 1) k' survivors per query (r = growth ratio, k' = rows
        // within 2 eps of the k-th): doubling keeps that at k' per panel (measured: r = 4, 8, 16 are slower).
        const int64_t len = panel == 0 ? first_panel : (panel == 1 && ratio == 2 && ix->panel_ratio < 2 ? 3 * j0 : (ratio - 1) * j0);
        const int64_t j1 = j0 + len < N ? j0 + len : N;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (ix->profile) {
            e0 = next_event(ix);
            e1 = next_event(ix);
            cudaEventRecord(e0, s);
        }
        KNN_CHECK(gemm_filter_launch(ix->plan, xq_h16, fmt_q, nb, nb_pad, ix->dp, ix->xb_h16, ix->shadow_fmt, N, ix->ynorm2, j0, j1,
                                     ix->metric, panel == 0, st, s));
        if (ix->profile) cudaEventRecord(e1, s);
        ix->st_gemm_launches++;
        KNN_CHECK(launch_tighten(st, W.eps.as<float>() + off, nb, k, 1, nullptr, d_overflow, s));
        j0 = j1;
        ++panel;
    }
    return KNN_OK;
}

// Finish phase of one batch: exact fp32 rescoring of every candidate at or above thr, then the sorted top-k.
// `lower` (optional) is a lower bound of the TRUE k-th best score per query obtained elsewhere (other shards):
// a row can only be in the global top-k if its approximate score is >= lower - eps.
int tensor_finish_batch(knn_index* ix, knn_index::TensorWs& W, int64_t off, int64_t nb, int k, int cap, const float* lower,
                        const float* neg_lower2, float* D, int64_t* I, int64_t id_base, cudaStream_t s) {
    const int largest = ix->metric == KNN_METRIC_INNER_PRODUCT;
    FilterState st = filter_state(W, off, cap);
    // the bound applied is max(lower, -neg_lower2) (either may be absent)
    if (lower) KNN_CHECK(launch_apply_lower(st.thr, W.eps.as<float>() + off, lower, neg_lower2, nb, s));
    if (ix->profile) cudaEventRecord(next_event_r(ix), s);
    KNN_CHECK(launch_rerank(W.xq_f32.as<float>() + off * ix->dp, W.xnorm2.as<float>() + off, nb, ix->dp, ix->xb_f32,
                            bf16_rows(ix), ix->ynorm2, ix->metric, st.cand_scores, st.cand_ids, st.counts, st.thr, cap, ix->ntotal, k,
                            ix->l2_blocked_rerank, s));
    if (ix->profile) cudaEventRecord(next_event_r(ix), s);
    KNN_CHECK(launch_select_final(st.cand_scores, st.cand_ids, st.counts, cap, 0, nb, k, largest, D, I, id_base, s));
    return KNN_OK;
}

int redo_overflowed(knn_index* ix, int64_t nq, int64_t qb, int64_t nbatches, const void* xq_dev, int qdt, int k, float* D,
                    int64_t* I, int64_t id_base, cudaStream_t s) {
    // A candidate list that ran past its capacity (heavily duplicated / clustered scores) is never truncated
    // silently: exactly the queries it happened to are redone with the exact scan and their rows replaced.
    std::vector<int> h_overflow(size_t(nbatches), 0);
    KNN_CHECK_CUDA(cudaMemcpyAsync(h_overflow.data(), ix->overflow.p, sizeof(int) * size_t(nbatches), cudaMemcpyDeviceToHost, s));
    KNN_CHECK_CUDA(cudaStreamSynchronize(s));
    std::vector<int> redo;
    std::vector<int> flags;
    for (int64_t b = 0; b < nbatches; ++b) {
        if (!h_overflow[size_t(b)]) continue;
        const int64_t q0 = b * qb;
        const int64_t nb = nq - q0 < qb ? nq - q0 : qb;
        ix->st_overflow_batches++;
        flags.resize(size_t(nb));
        KNN_CHECK_CUDA(cudaMemcpyAsync(flags.data(), ix->ovf_q.as<int>() + q0, sizeof(int) * size_t(nb), cudaMemcpyDeviceToHost, s));
        KNN_CHECK_CUDA(cudaStreamSynchronize(s));
        for (int64_t i = 0; i < nb; ++i)
            if (flags[size_t(i)]) redo.push_back(int(q0 + i));
    }
    ix->st_overflow_queries += (long long)redo.size();
    const int64_t chunk = 1024;
    for (size_t c0 = 0; c0 < redo.size(); c0 += size_t(chunk)) {
        const int64_t n = int64_t(std::min(redo.size() - c0, size_t(chunk)));
        KNN_CHECK(ix->ovf_idx.ensure(sizeof(int) * size_t(chunk)));
        KNN_CHECK(ix->ovf_x.ensure(sizeof(float) * size_t(chunk) * ix->d));
        KNN_CHECK(ix->ovf_D.ensure(sizeof(float) * size_t(chunk) * k));
        KNN_CHECK(ix->ovf_I.ensure(sizeof(int64_t) * size_t(chunk) * k));
        KNN_CHECK_CUDA(cudaMemcpyAsync(ix->ovf_idx.p, redo.data() + c0, sizeof(int) * size_t(n), cudaMemcpyHostToDevice, s));
        // the flagged rows are gathered as fp32 (exact for 16-bit queries): the scan sees the values it would have seen
        KNN_CHECK(launch_gather_rows(xq_dev, qdt, ix->d, ix->ovf_idx.as<int>(), n, ix->ovf_x.as<float>(), s));
        KNN_CHECK(search_exact(ix, n, ix->ovf_x.p, KNN_DTYPE_F32, k, ix->ovf_D.as<float>(), ix->ovf_I.as<int64_t>(), id_base, s));
        KNN_CHECK(launch_scatter_results(ix->ovf_D.as<float>(), ix->ovf_I.as<int64_t>(), ix->ovf_idx.as<int>(), n, k, D, I, s));
        KNN_CHECK_CUDA(cudaStreamSynchronize(s));  // `redo` chunk consumed
    }
    return KNN_OK;
}

// Host-pointer search, pipelined (knn_index_search).  The reference's drivers hand index.search pageable numpy arrays
// (cath/search.py:24, seqvec_search/main.py:45): per query batch the queries are staged into a pinned bounce buffer by
// the calling thread, cross PCIe on a copy stream while the previous batch is on the tensor cores, and the batch's
// (D, I) rows travel back on a second copy stream while the next batch is filtered.  Pinned caller memory is DMA'd
// directly.  Everything is enqueued asynchronously; the host only ever waits for the slot it is about to reuse.
struct HostPipe {
    knn_index* ix;
    const void* xq;
    int qdt;  // element type of xq: the bounce buffers and copies move the caller's bytes as they are
    float* D;
    int64_t* I;
    int k;
    bool in_pinned, out_pinned;
    int64_t slot_q0[2] = {-1, -1}, slot_nb[2] = {0, 0};

    int init(int64_t qb) {
        const size_t in_bytes = size_t(qb) * ix->d * dtype_size(qdt);
        for (int w = 0; w < 2; ++w) {
            KNN_CHECK(ix->hp_xq[w].ensure(in_bytes));
            KNN_CHECK(ix->hp_D[w].ensure(size_t(qb) * k * sizeof(float)));
            KNN_CHECK(ix->hp_I[w].ensure(size_t(qb) * k * sizeof(int64_t)));
            if (!in_pinned) KNN_CHECK(ix->hp_pin_xq[w].ensure(in_bytes));
            if (!out_pinned) {
                KNN_CHECK(ix->hp_pin_D[w].ensure(size_t(qb) * k * sizeof(float)));
                KNN_CHECK(ix->hp_pin_I[w].ensure(size_t(qb) * k * sizeof(int64_t)));
            }
        }
        return KNN_OK;
    }
    // the results of the batch that last used slot w are in the caller's memory; the slot is free
    int drain(int w) {
        if (slot_q0[w] < 0) return KNN_OK;
        KNN_CHECK_CUDA(cudaEventSynchronize(ix->hp_out_done[w]));
        if (!out_pinned) {
            host_copy(D + slot_q0[w] * k, ix->hp_pin_D[w].p, size_t(slot_nb[w]) * k * sizeof(float));
            host_copy(I + slot_q0[w] * k, ix->hp_pin_I[w].p, size_t(slot_nb[w]) * k * sizeof(int64_t));
        }
        slot_q0[w] = -1;
        return KNN_OK;
    }
    // before batch b: its queries on the way to the device, `s` ordered behind the copy.  The input slot is free as
    // soon as the filter of batch b - 2 has read it - NOT when that batch's results are home: its finish phase runs at
    // low priority under the filter of batch b - 1, and staging the next queries must not wait for it.
    int acquire(int64_t b, int64_t q0, int64_t nb, cudaStream_t s, const void** xq_b, float** D_b, int64_t** I_b) {
        const int w = int(b & 1);
        if (b >= 2) KNN_CHECK_CUDA(cudaEventSynchronize(ix->hp_in_free[w]));
        const size_t bytes = size_t(nb) * ix->d * dtype_size(qdt);
        const void* src = row_at(xq, q0, ix->d, qdt);
        if (!in_pinned) {
            host_copy(ix->hp_pin_xq[w].p, src, bytes);
            src = ix->hp_pin_xq[w].p;
        }
        KNN_CHECK_CUDA(cudaMemcpyAsync(ix->hp_xq[w].p, src, bytes, cudaMemcpyHostToDevice, ix->copy_in));
        KNN_CHECK_CUDA(cudaEventRecord(ix->hp_in_ready[w], ix->copy_in));
        KNN_CHECK_CUDA(cudaStreamWaitEvent(s, ix->hp_in_ready[w], 0));
        *xq_b = ix->hp_xq[w].p;
        *D_b = ix->hp_D[w].as<float>();
        *I_b = ix->hp_I[w].as<int64_t>();
        return KNN_OK;
    }
    // after the filter of batch b was enqueued on `s`: the input slot can be refilled once it has run
    int filtered(int64_t b, cudaStream_t s) {
        KNN_CHECK_CUDA(cudaEventRecord(ix->hp_in_free[int(b & 1)], s));
        return KNN_OK;
    }
    // before the finish phase of batch b is enqueued on `fs`: the output slot's previous rows (batch b - 2) are home
    int before_finish(int64_t b) { return drain(int(b & 1)); }
    // after the finish phase of batch b was enqueued on `fs`: its rows on the way back
    int release(int64_t b, int64_t q0, int64_t nb, cudaStream_t fs) {
        const int w = int(b & 1);
        KNN_CHECK_CUDA(cudaEventRecord(ix->hp_computed[w], fs));
        KNN_CHECK_CUDA(cudaStreamWaitEvent(ix->copy_out, ix->hp_computed[w], 0));
        float* dD = out_pinned ? D + q0 * k : ix->hp_pin_D[w].as<float>();
        int64_t* dI = out_pinned ? I + q0 * k : ix->hp_pin_I[w].as<int64_t>();
        KNN_CHECK_CUDA(cudaMemcpyAsync(dD, ix->hp_D[w].p, size_t(nb) * k * sizeof(float), cudaMemcpyDeviceToHost, ix->copy_out));
        KNN_CHECK_CUDA(cudaMemcpyAsync(dI, ix->hp_I[w].p, size_t(nb) * k * sizeof(int64_t), cudaMemcpyDeviceToHost, ix->copy_out));
        KNN_CHECK_CUDA(cudaEventRecord(ix->hp_out_done[w], ix->copy_out));
        slot_q0[w] = q0;
        slot_nb[w] = nb;
        return KNN_OK;
    }
    int finish() {
        KNN_CHECK(drain(0));
        KNN_CHECK(drain(1));
        return KNN_OK;
    }
};

// Overflow repair of a host-pointer search: the flagged queries (rare: heavily duplicated rows, out-of-range data) are
// uploaded again, answered by the exact scan and written into the caller's rows.
int redo_overflowed_host(knn_index* ix, int64_t nq, int64_t qb, int64_t nbatches, const void* xq, int qdt, int k, float* D,
                         int64_t* I, cudaStream_t s) {
    std::vector<int> h_overflow(size_t(nbatches), 0);
    KNN_CHECK_CUDA(cudaMemcpyAsync(h_overflow.data(), ix->overflow.p, sizeof(int) * size_t(nbatches), cudaMemcpyDeviceToHost, s));
    KNN_CHECK_CUDA(cudaStreamSynchronize(s));
    std::vector<int> redo, flags;
    for (int64_t b = 0; b < nbatches; ++b) {
        if (!h_overflow[size_t(b)]) continue;
        const int64_t q0 = b * qb;
        const int64_t nb = nq - q0 < qb ? nq - q0 : qb;
        ix->st_overflow_batches++;
        flags.resize(size_t(nb));
        KNN_CHECK_CUDA(cudaMemcpyAsync(flags.data(), ix->ovf_q.as<int>() + q0, sizeof(int) * size_t(nb), cudaMemcpyDeviceToHost, s));
        KNN_CHECK_CUDA(cudaStreamSynchronize(s));
        for (int64_t i = 0; i < nb; ++i)
            if (flags[size_t(i)]) redo.push_back(int(q0 + i));
    }
    ix->st_overflow_queries += (long long)redo.size();
    const int64_t chunk = 1024;
    const size_t row_bytes = size_t(ix->d) * dtype_size(qdt);  // the rows travel in the caller's element type
    std::vector<char> hx;
    std::vector<float> hD;
    std::vector<int64_t> hI;
    for (size_t c0 = 0; c0 < redo.size(); c0 += size_t(chunk)) {
        const int64_t n = int64_t(std::min(redo.size() - c0, size_t(chunk)));
        KNN_CHECK(ix->ovf_x.ensure(row_bytes * size_t(chunk)));
        KNN_CHECK(ix->ovf_D.ensure(sizeof(float) * size_t(chunk) * k));
        KNN_CHECK(ix->ovf_I.ensure(sizeof(int64_t) * size_t(chunk) * k));
        hx.resize(size_t(n) * row_bytes);
        for (int64_t i = 0; i < n; ++i) memcpy(hx.data() + i * row_bytes, row_at(xq, redo[c0 + size_t(i)], ix->d, qdt), row_bytes);
        KNN_CHECK_CUDA(cudaMemcpyAsync(ix->ovf_x.p, hx.data(), hx.size(), cudaMemcpyHostToDevice, s));
        KNN_CHECK(search_exact(ix, n, ix->ovf_x.p, qdt, k, ix->ovf_D.as<float>(), ix->ovf_I.as<int64_t>(), 0, s));
        hD.resize(size_t(n) * k);
        hI.resize(size_t(n) * k);
        KNN_CHECK_CUDA(cudaMemcpyAsync(hD.data(), ix->ovf_D.p, sizeof(float) * hD.size(), cudaMemcpyDeviceToHost, s));
        KNN_CHECK_CUDA(cudaMemcpyAsync(hI.data(), ix->ovf_I.p, sizeof(int64_t) * hI.size(), cudaMemcpyDeviceToHost, s));
        KNN_CHECK_CUDA(cudaStreamSynchronize(s));
        for (int64_t i = 0; i < n; ++i) {
            memcpy(D + int64_t(redo[c0 + size_t(i)]) * k, hD.data() + i * k, sizeof(float) * k);
            memcpy(I + int64_t(redo[c0 + size_t(i)]) * k, hI.data() + i * k, sizeof(int64_t) * k);
        }
    }
    return KNN_OK;
}

// `hp` (host-pointer search): xq_dev / D / I are then HOST pointers that only the pipe touches.
int search_tensor(knn_index* ix, int64_t nq, const void* xq_dev, int qdt, int k, float* D, int64_t* I, int64_t id_base,
                  cudaStream_t s, HostPipe* hp = nullptr) {
    const int cap = candidate_capacity(k, ix->ntotal, ix->dense_small_db != 0);
    int64_t qb = ix->query_batch;
    if (qb > nq) qb = nq;
    // A call that fits one batch has nothing to overlap its finish phase with.  Where that phase is heavy (k >= 256:
    // ~k rows of 4 KB gathered per query) and there are enough queries to keep the GEMM tiles full, the call is cut
    // into up to four batches so that rescoring runs under the next batch's filter (C2: 14,433 queries, k = 1000).
    if (ix->overlap_finish && ix->split_single_batch && qb == nq && k >= 256 && nq >= 4096) {
        const int64_t parts = std::min<int64_t>(4, nq / 2048);
        qb = (nq + parts - 1) / parts;
    }
    qb = round_up(qb, 256);
    const int64_t nbatches = (nq + qb - 1) / qb;
    // The finish phase of a batch (exact rescoring + final select: HBM gathers and shared-memory sorts) runs on a
    // side stream under the tensor-core filter of the next batch, which leaves HBM and most of every SM's registers
    // idle; the two batches live in two workspaces.  One batch: nothing to overlap with.
    const bool overlap = ix->overlap_finish && nbatches > 1;
    KNN_CHECK(tensor_ws_ensure(ix->ws1[0], qb, ix->dp, cap));
    if (overlap) KNN_CHECK(tensor_ws_ensure(ix->ws1[1], qb, ix->dp, cap));
    KNN_CHECK(ix->overflow.ensure(sizeof(int) * size_t(nbatches)));
    KNN_CHECK(ix->ovf_q.ensure(sizeof(int) * size_t(nq)));
    KNN_CHECK(tensor_prepare(ix));
    if (hp) KNN_CHECK(hp->init(qb));
    KNN_CHECK_CUDA(cudaMemsetAsync(ix->overflow.p, 0, sizeof(int) * size_t(nbatches), s));
    // a previous call's side-stream work (possibly issued from another stream) still owns the workspaces
    KNN_CHECK_CUDA(cudaStreamWaitEvent(s, ix->ev_finished[0], 0));
    KNN_CHECK_CUDA(cudaStreamWaitEvent(s, ix->ev_finished[1], 0));
    // Overlapped: the filter phase moves to an internal HIGH-priority stream and the finish phase runs on a
    // LOW-priority one.  Without that the thousands of short rescoring CTAs, enqueued first, are dispatched ahead of
    // the next GEMM launches and the two phases merely swap places; with it a GEMM CTA takes the first slot that
    // frees up and rescoring fills what the resident GEMM CTAs leave (registers, ~64 KB of shared memory, HBM).
    cudaStream_t caller = s;
    if (overlap) {
        KNN_CHECK_CUDA(cudaEventRecord(ix->ev_fork, caller));
        KNN_CHECK_CUDA(cudaStreamWaitEvent(ix->hi, ix->ev_fork, 0));
        s = ix->hi;
    }
    for (int64_t b = 0; b < nbatches; ++b) {
        const int64_t q0 = b * qb;
        const int64_t nb = nq - q0 < qb ? nq - q0 : qb;
        const int w = overlap ? int(b & 1) : 0;
        const void* xq_b = hp ? nullptr : row_at(xq_dev, q0, ix->d, qdt);
        float* D_b = hp ? nullptr : D + q0 * k;
        int64_t* I_b = hp ? nullptr : I + q0 * k;
        if (hp) KNN_CHECK(hp->acquire(b, q0, nb, s, &xq_b, &D_b, &I_b));
        if (overlap && b >= 2) KNN_CHECK_CUDA(cudaStreamWaitEvent(s, ix->ev_finished[w], 0));  // ws1[w] is free again
        KNN_CHECK(tensor_filter_batch(ix, ix->ws1[w], 0, nb, xq_b, qdt, k, cap, ix->overflow.as<int>() + b, ix->ovf_q.as<int>() + q0, s));
        if (hp) {
            KNN_CHECK(hp->filtered(b, s));
            KNN_CHECK(hp->before_finish(b));
        }
        cudaStream_t fs = s;
        if (overlap) {
            fs = ix->side;
            KNN_CHECK_CUDA(cudaEventRecord(ix->ev_filtered[w], s));
            KNN_CHECK_CUDA(cudaStreamWaitEvent(fs, ix->ev_filtered[w], 0));
        }
        KNN_CHECK(tensor_finish_batch(ix, ix->ws1[w], 0, nb, k, cap, nullptr, nullptr, D_b, I_b, id_base, fs));
        if (overlap) KNN_CHECK_CUDA(cudaEventRecord(ix->ev_finished[w], fs));
        if (hp) KNN_CHECK(hp->release(b, q0, nb, fs));
    }
    if (overlap) {  // the caller's stream sees every result (and the per-batch overflow flags)
        KNN_CHECK_CUDA(cudaEventRecord(ix->ev_join, s));
        s = caller;
        KNN_CHECK_CUDA(cudaStreamWaitEvent(s, ix->ev_join, 0));
        KNN_CHECK_CUDA(cudaStreamWaitEvent(s, ix->ev_finished[0], 0));
        KNN_CHECK_CUDA(cudaStreamWaitEvent(s, ix->ev_finished[1], 0));
    }
    if (hp) {
        KNN_CHECK(hp->finish());
        return redo_overflowed_host(ix, nq, qb, nbatches, xq_dev, qdt, k, D, I, s);
    }
    return redo_overflowed(ix, nq, qb, nbatches, xq_dev, qdt, k, D, I, id_base, s);
}

bool use_tensor_path(const knn_index* ix, int64_t nq, int k) {
    bool tensor = ix->path_param == 2 || (ix->path_param == 0 && nq >= ix->tensor_min_nq && ix->ntotal >= ix->tensor_min_n);
    if (ix->ntotal < k) tensor = false;
    return tensor;
}

int search_dev_impl(knn_index* ix, int64_t nq, const void* xq_dev, int qdt, int64_t k64, float* D, int64_t* I, int64_t id_base,
                    cudaStream_t s, HostPipe* hp = nullptr) {
    if (nq < 0 || k64 <= 0 || (nq > 0 && (!xq_dev || !D || !I))) {
        set_error("search: invalid arguments (nq=%lld, k=%lld)", (long long)nq, (long long)k64);
        return KNN_ERR_INVALID;
    }
    KNN_CHECK(check_dtype(qdt, "search"));
    if (k64 > KNN_MAX_K) {
        set_error("search: k=%lld exceeds KNN_MAX_K=%d", (long long)k64, KNN_MAX_K);
        return KNN_ERR_LIMIT;
    }
    if (nq == 0) return KNN_OK;
    KNN_CHECK_CUDA(cudaStreamWaitEvent(s, ix->add_event, 0));
    const int k = int(k64);
    const long long launches0 = g_launches.load();
    ix->st_gemm_launches = 0;
    ix->st_gemm_ms = 0;
    ix->st_rerank_ms = 0;
    ix->ev_used_r = 0;
    ix->st_overflow_batches = 0;
    ix->st_overflow_queries = 0;
    ix->ev_used = 0;
    int rc;
    if (ix->ntotal == 0) {
        // nothing to search: all padding (select over an empty list)
        KNN_CHECK(ix->lists_s.ensure(16));
        KNN_CHECK(ix->lists_i.ensure(16));
        rc = launch_select_final(ix->lists_s.as<float>(), ix->lists_i.as<uint32_t>(), nullptr, 0, 0, nq, k,
                                 ix->metric == KNN_METRIC_INNER_PRODUCT, D, I, id_base, s);
        ix->last_path = 1;
    } else {
        const bool tensor = use_tensor_path(ix, nq, k);
        ix->last_path = tensor ? 2 : 1;
        if (tensor) KNN_CHECK(prepare_shadow(ix, k, s));
        if (hp && !tensor) {
            set_error("internal: host pipe on the exact path");
            return KNN_ERR_INVALID;
        }
        rc = tensor ? search_tensor(ix, nq, xq_dev, qdt, k, D, I, id_base, s, hp)
                    : search_exact(ix, nq, xq_dev, qdt, k, D, I, id_base, s);
    }
    if (rc != KNN_OK) return rc;
    KNN_CHECK_CUDA(cudaEventRecord(ix->search_event, s));
    if (ix->profile && ix->ev_used) {
        KNN_CHECK_CUDA(cudaStreamSynchronize(s));
        collect_profile(ix);
    }
    ix->st_launches = g_launches.load() - launches0;
    return KNN_OK;
}

}  // namespace

// =============================================================================================
extern "C" {

const char* knn_last_error(void) { return g_error.c_str(); }

int knn_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int64_t knn_kernel_launches(void) { return g_launches.load(); }

int knn_normalize_l2_dev(float* x_dev, int64_t n, int64_t d, void* stream) {
    if (n < 0 || d <= 0 || (n > 0 && !x_dev)) {
        set_error("normalize_l2: invalid arguments");
        return KNN_ERR_INVALID;
    }
    PtrDeviceGuard g(x_dev);
    return launch_normalize_l2(x_dev, n, d, static_cast<cudaStream_t>(stream));
}

int knn_normalize_l2(float* x, int64_t n, int64_t d, int device) {
    if (n < 0 || d <= 0 || (n > 0 && !x)) {
        set_error("normalize_l2: invalid arguments");
        return KNN_ERR_INVALID;
    }
    if (n == 0) return KNN_OK;
    DeviceGuard g(device);
    if (!g.ok) {
        set_error("normalize_l2: cannot select CUDA device %d (no CPU fallback)", device);
        return KNN_ERR_CUDA;
    }
    // stream the matrix through a bounded device buffer
    const int64_t rows_per = std::max<int64_t>(1, (int64_t(256) << 20) / (d * 4));
    float* buf = nullptr;
    const int64_t rows_alloc = n < rows_per ? n : rows_per;
    KNN_CHECK_CUDA(cudaMalloc(&buf, size_t(rows_alloc) * d * sizeof(float)));
    int rc = KNN_OK;
    for (int64_t r0 = 0; r0 < n && rc == KNN_OK; r0 += rows_per) {
        const int64_t nr = n - r0 < rows_per ? n - r0 : rows_per;
        cudaError_t e = cudaMemcpy(buf, x + r0 * d, size_t(nr) * d * sizeof(float), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) {
            rc = launch_normalize_l2(buf, nr, d, nullptr);
            if (rc == KNN_OK) e = cudaMemcpy(x + r0 * d, buf, size_t(nr) * d * sizeof(float), cudaMemcpyDeviceToHost);
        }
        if (e != cudaSuccess) {
            set_error("normalize_l2: copy failed: %s", cudaGetErrorString(e));
            rc = KNN_ERR_CUDA;
        }
    }
    cudaFree(buf);
    return rc;
}

int knn_index_create(knn_index** out, int d, int metric, int device, unsigned flags) {
    if (!out || d <= 0 || (metric != KNN_METRIC_INNER_PRODUCT && metric != KNN_METRIC_L2)) {
        set_error("index_create: invalid arguments (d=%d, metric=%d)", d, metric);
        return KNN_ERR_INVALID;
    }
    int ndev = knn_device_count();
    if (device < 0 || device >= ndev) {
        set_error("index_create: CUDA device %d not available (%d visible); this library has no CPU fallback", device, ndev);
        return KNN_ERR_CUDA;
    }
    DeviceGuard g(device);
    if (!g.ok) {
        set_error("index_create: cannot select device %d", device);
        return KNN_ERR_CUDA;
    }
    knn_index* ix = new knn_index();
    ix->d = d;
    ix->dp = int(round_up(d, kDimAlign));
    ix->metric = metric;
    ix->device = device;
    ix->flags = flags;
    cudaError_t e = cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->add_event, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->search_event, cudaEventDisableTiming);
    int prio_least = 0, prio_greatest = 0;
    if (e == cudaSuccess) e = cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ix->side, cudaStreamNonBlocking, prio_least);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&ix->hi, cudaStreamNonBlocking, prio_greatest);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->ev_join, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ix->copy_in, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ix->copy_out, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaEventCreateWithFlags(&ix->hp_in_ready[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->hp_out_done[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->hp_computed[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->hp_in_free[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->stage_free[i], cudaEventDisableTiming);
    }
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaEventCreateWithFlags(&ix->ev_filtered[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->ev_finished[i], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaMalloc(&ix->stats, sizeof(DbStats));
    if (e == cudaSuccess) e = cudaMemset(ix->stats, 0, sizeof(DbStats));
    if (e != cudaSuccess) {
        set_error("index_create: %s", cudaGetErrorString(e));
        delete ix;
        return KNN_ERR_CUDA;
    }
    *out = ix;
    return KNN_OK;
}

int knn_index_free(knn_index* ix) {
    if (!ix) return KNN_OK;
    DeviceGuard g(ix->device);
    cudaStreamSynchronize(ix->stream);
    if (ix->side) cudaStreamSynchronize(ix->side);
    if (ix->hi) cudaStreamSynchronize(ix->hi);
    for (DevBuf* b : {&ix->stage, &ix->xq_f32, &ix->xnorm2, &ix->eps, &ix->scores, &ix->lists_s, &ix->lists_i,
                      &ix->overflow, &ix->ovf_q, &ix->ovf_idx, &ix->ovf_x, &ix->ovf_D, &ix->ovf_I, &ix->h_xq, &ix->h_D, &ix->h_I})
        b->release();
    for (int i = 0; i < 2; ++i) {
        ix->hp_xq[i].release(); ix->hp_D[i].release(); ix->hp_I[i].release();
        ix->hp_pin_xq[i].release(); ix->hp_pin_D[i].release(); ix->hp_pin_I[i].release();
        for (cudaEvent_t e : {ix->hp_in_ready[i], ix->hp_out_done[i], ix->hp_computed[i], ix->stage_free[i], ix->hp_in_free[i]})
            if (e) cudaEventDestroy(e);
    }
    ix->stage2.release();
    if (ix->copy_in) cudaStreamDestroy(ix->copy_in);
    if (ix->copy_out) cudaStreamDestroy(ix->copy_out);
    for (knn_index::TensorWs* W : {&ix->ws1[0], &ix->ws1[1], &ix->ws2})
        for (DevBuf* b : {&W->xq_f32, &W->xq_h16, &W->xnorm2, &W->eps, &W->thr, &W->counts, &W->cand_s, &W->cand_i}) b->release();
    if (ix->xb_f32) cudaFree(ix->xb_f32);
    if (ix->xb_h16) cudaFree(ix->xb_h16);
    if (ix->ynorm2) cudaFree(ix->ynorm2);
    if (ix->stats) cudaFree(ix->stats);
    for (cudaEvent_t e : ix->ev_pool) cudaEventDestroy(e);
    for (cudaEvent_t e : ix->ev_pool_r) cudaEventDestroy(e);
    if (ix->add_event) cudaEventDestroy(ix->add_event);
    if (ix->search_event) cudaEventDestroy(ix->search_event);
    for (int i = 0; i < 2; ++i) {
        if (ix->ev_filtered[i]) cudaEventDestroy(ix->ev_filtered[i]);
        if (ix->ev_finished[i]) cudaEventDestroy(ix->ev_finished[i]);
    }
    if (ix->side) cudaStreamDestroy(ix->side);
    if (ix->hi) cudaStreamDestroy(ix->hi);
    if (ix->ev_fork) cudaEventDestroy(ix->ev_fork);
    if (ix->ev_join) cudaEventDestroy(ix->ev_join);
    if (ix->plan) gemm_plan_destroy(ix->plan);
    if (ix->stream) cudaStreamDestroy(ix->stream);
    delete ix;
    return KNN_OK;
}

int knn_index_reset(knn_index* ix) {
    if (!ix) return KNN_ERR_INVALID;
    DeviceGuard g(ix->device);
    ix->ntotal = 0;
    ix->stats_dirty = false;
    ix->fp16_unfit = false;
    KNN_CHECK_CUDA(cudaStreamWaitEvent(ix->stream, ix->search_event, 0));
    KNN_CHECK_CUDA(cudaStreamWaitEvent(ix->stream, ix->add_event, 0));
    KNN_CHECK_CUDA(cudaMemsetAsync(ix->stats, 0, sizeof(DbStats), ix->stream));
    KNN_CHECK_CUDA(cudaStreamSynchronize(ix->stream));
    return KNN_OK;
}

int knn_index_reserve(knn_index* ix, int64_t n) {
    if (!ix || n < 0) return KNN_ERR_INVALID;
    DeviceGuard g(ix->device);
    // exact size: reserve is how large databases avoid the 1.5x growth slack
    return grow(ix, n, /*exact=*/true);
}

int knn_index_add_typed_dev(knn_index* ix, int64_t n, const void* x_dev, int dtype, void* stream) {
    if (!ix || n < 0 || (n > 0 && !x_dev)) {
        set_error("add: invalid arguments");
        return KNN_ERR_INVALID;
    }
    KNN_CHECK(check_dtype(dtype, "add"));
    if (n == 0) return KNN_OK;
    DeviceGuard g(ix->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    KNN_CHECK(grow(ix, ix->ntotal + n));
    // a search still in flight on another stream may be rewriting the shadow rows and their statistics
    KNN_CHECK_CUDA(cudaStreamWaitEvent(s, ix->search_event, 0));
    const int64_t r0 = ix->ntotal;
    if (r0 == 0) {  // an empty index takes the format its expected size asks for; later rows follow the rows already there
        const ShadowChoice c = desired_shadow(ix, 0, std::max<int64_t>(ix->capacity, n));
        ix->shadow_fmt = c.fmt;
        ix->shadow_mbits = c.mbits;
    }
    KNN_CHECK(launch_ingest(x_dev, dtype, ix->d, n, ix->d, ix->dp, ix->xb_f32 ? ix->xb_f32 + r0 * ix->dp : nullptr,
                            ix->xb_h16 + r0 * ix->dp, ix->shadow_fmt, ix->shadow_mbits, bf16_only(ix), ix->ynorm2 + r0,
                            ix->stats, s));
    KNN_CHECK_CUDA(cudaEventRecord(ix->add_event, s));
    ix->ntotal += n;
    ix->stats_dirty = true;
    return KNN_OK;
}

int knn_index_add_dev(knn_index* ix, int64_t n, const float* x_dev, void* stream) {
    return knn_index_add_typed_dev(ix, n, x_dev, KNN_DTYPE_F32, stream);
}

int knn_index_add_typed(knn_index* ix, int64_t n, const void* x, int dtype) {
    if (!ix || n < 0 || (n > 0 && !x)) {
        set_error("add: invalid arguments");
        return KNN_ERR_INVALID;
    }
    KNN_CHECK(check_dtype(dtype, "add"));
    if (n == 0) return KNN_OK;
    DeviceGuard g(ix->device);
    KNN_CHECK(grow(ix, ix->ntotal + n));
    // chunks of <= 64 MiB through two staging buffers: the H2D copy of chunk i + 1 (copy stream) runs while chunk i is
    // ingested (index stream); pageable caller memory goes through the driver's own bounce buffers.  The chunks hold the
    // caller's bytes as they are: 16-bit rows are converted by the ingest kernel, not before the copy.
    const size_t row_bytes = size_t(ix->d) * dtype_size(dtype);
    const int64_t rows_per = std::max<int64_t>(1, (int64_t(64) << 20) / int64_t(row_bytes));
    const size_t stage_bytes = size_t(n < rows_per ? n : rows_per) * row_bytes;
    KNN_CHECK(ix->stage.ensure(stage_bytes));
    if (n > rows_per) KNN_CHECK(ix->stage2.ensure(stage_bytes));
    int64_t c = 0;
    auto add_chunks = [&]() -> int {
        for (int64_t r0 = 0; r0 < n; r0 += rows_per, ++c) {
            const int64_t nr = n - r0 < rows_per ? n - r0 : rows_per;
            const int w = int(c & 1);
            void* st = (w ? ix->stage2 : ix->stage).p;
            if (c >= 2) KNN_CHECK_CUDA(cudaEventSynchronize(ix->stage_free[w]));  // the ingest that read this buffer is done
            KNN_CHECK_CUDA(cudaMemcpyAsync(st, row_at(x, r0, ix->d, dtype), size_t(nr) * row_bytes, cudaMemcpyHostToDevice, ix->copy_in));
            KNN_CHECK_CUDA(cudaEventRecord(ix->hp_in_ready[w], ix->copy_in));
            KNN_CHECK_CUDA(cudaStreamWaitEvent(ix->stream, ix->hp_in_ready[w], 0));
            KNN_CHECK(knn_index_add_typed_dev(ix, nr, st, dtype, ix->stream));
            KNN_CHECK_CUDA(cudaEventRecord(ix->stage_free[w], ix->stream));
        }
        return KNN_OK;
    };
    const int rc = add_chunks();
    // `add` copies (faiss semantics): the caller may reuse x once this returns - also when it returns an error
    if (rc != KNN_OK) {
        cudaDeviceSynchronize();
        return rc;
    }
    KNN_CHECK_CUDA(cudaStreamSynchronize(ix->stream));
    return KNN_OK;
}

int knn_index_add(knn_index* ix, int64_t n, const float* x) { return knn_index_add_typed(ix, n, x, KNN_DTYPE_F32); }

int64_t knn_index_ntotal(const knn_index* ix) { return ix ? ix->ntotal : -1; }
int knn_index_d(const knn_index* ix) { return ix ? ix->d : -1; }
int knn_index_metric(const knn_index* ix) { return ix ? ix->metric : -1; }

int knn_index_search_typed_dev(knn_index* ix, int64_t nq, const void* xq_dev, int dtype, int64_t k, float* D_dev,
                               int64_t* I_dev, int64_t id_base, void* stream) {
    if (!ix) {
        set_error("search: null index");
        return KNN_ERR_INVALID;
    }
    DeviceGuard g(ix->device);
    return search_dev_impl(ix, nq, xq_dev, dtype, k, D_dev, I_dev, id_base, static_cast<cudaStream_t>(stream));
}

int knn_index_search_dev(knn_index* ix, int64_t nq, const float* xq_dev, int64_t k, float* D_dev, int64_t* I_dev,
                         int64_t id_base, void* stream) {
    return knn_index_search_typed_dev(ix, nq, xq_dev, KNN_DTYPE_F32, k, D_dev, I_dev, id_base, stream);
}

int knn_index_search_typed(knn_index* ix, int64_t nq, const void* xq, int dtype, int64_t k, float* D, int64_t* I) {
    if (!ix || nq < 0 || k <= 0 || (nq > 0 && (!xq || !D || !I))) {
        set_error("search: invalid arguments (nq=%lld, k=%lld)", (long long)nq, (long long)k);
        return KNN_ERR_INVALID;
    }
    KNN_CHECK(check_dtype(dtype, "search"));
    if (k > KNN_MAX_K) {
        set_error("search: k=%lld exceeds KNN_MAX_K=%d", (long long)k, KNN_MAX_K);
        return KNN_ERR_LIMIT;
    }
    if (nq == 0) return KNN_OK;
    DeviceGuard g(ix->device);
    if (ix->ntotal > 0 && use_tensor_path(ix, nq, int(k))) {
        // tensor path: one pipelined pass over the query batches (copies under compute, see HostPipe)
        HostPipe hp{ix, xq, dtype, D, I, int(k), host_pointer_is_pinned(xq), host_pointer_is_pinned(D) && host_pointer_is_pinned(I)};
        const int rc = search_dev_impl(ix, nq, xq, dtype, k, D, I, 0, ix->stream, &hp);
        if (rc != KNN_OK) {
            // copies into / out of the caller's arrays may still be in flight on the copy streams: nothing may touch
            // the caller's memory once this call has returned, error or not
            cudaDeviceSynchronize();
            return rc;
        }
        KNN_CHECK_CUDA(cudaStreamSynchronize(ix->stream));
        return KNN_OK;
    }
    // exact path (small databases / few queries): host batches bound the device staging buffers; each is
    // H2D -> search -> D2H on one stream
    const int64_t hb = 65536;
    const int64_t nb_max = nq < hb ? nq : hb;
    const size_t row_bytes = size_t(ix->d) * dtype_size(dtype);  // queries are staged in the caller's element type
    KNN_CHECK(ix->h_xq.ensure(size_t(nb_max) * row_bytes));
    KNN_CHECK(ix->h_D.ensure(size_t(nb_max) * k * sizeof(float)));
    KNN_CHECK(ix->h_I.ensure(size_t(nb_max) * k * sizeof(int64_t)));
    long long launches = 0, gemm_launches = 0, overflow = 0, overflow_q = 0;
    double gemm_ms = 0;
    for (int64_t q0 = 0; q0 < nq; q0 += hb) {
        const int64_t nb = nq - q0 < hb ? nq - q0 : hb;
        KNN_CHECK_CUDA(cudaMemcpyAsync(ix->h_xq.p, row_at(xq, q0, ix->d, dtype), size_t(nb) * row_bytes, cudaMemcpyHostToDevice, ix->stream));
        KNN_CHECK(search_dev_impl(ix, nb, ix->h_xq.p, dtype, k, ix->h_D.as<float>(), ix->h_I.as<int64_t>(), 0, ix->stream));
        KNN_CHECK_CUDA(cudaMemcpyAsync(D + q0 * k, ix->h_D.p, size_t(nb) * k * sizeof(float), cudaMemcpyDeviceToHost, ix->stream));
        KNN_CHECK_CUDA(cudaMemcpyAsync(I + q0 * k, ix->h_I.p, size_t(nb) * k * sizeof(int64_t), cudaMemcpyDeviceToHost, ix->stream));
        KNN_CHECK_CUDA(cudaStreamSynchronize(ix->stream));
        launches += ix->st_launches;
        gemm_launches += ix->st_gemm_launches;
        gemm_ms += ix->st_gemm_ms;
        overflow += ix->st_overflow_batches;
        overflow_q += ix->st_overflow_queries;
    }
    ix->st_launches = launches;
    ix->st_gemm_launches = gemm_launches;
    ix->st_gemm_ms = gemm_ms;
    ix->st_overflow_batches = overflow;
    ix->st_overflow_queries = overflow_q;
    return KNN_OK;
}

int knn_index_search(knn_index* ix, int64_t nq, const float* xq, int64_t k, float* D, int64_t* I) {
    return knn_index_search_typed(ix, nq, xq, KNN_DTYPE_F32, k, D, I);
}

// ---- two-phase (row-sharded) search ---------------------------------------------------------
// begin -> per batch: filter_batch ... (caller combines the bounds of all shards) ... finish_batch -> end.
// The batch-wise calls let the caller run exchange + finish of batch b on another stream under the filter of batch
// b + 1 (knn_b200/distributed.py); knn_index_search_filter_dev / _finish_dev are the all-batches-at-once form.
static int two_phase_begin(knn_index* ix, int64_t nq, const void* xq_dev, int qdt, int64_t k64, cudaStream_t s, const char* who) {
    if (!ix || nq <= 0 || k64 <= 0 || !xq_dev) {
        set_error("%s: invalid arguments", who);
        return KNN_ERR_INVALID;
    }
    KNN_CHECK(check_dtype(qdt, who));
    if (k64 > KNN_MAX_K) {
        set_error("%s: k=%lld exceeds KNN_MAX_K=%d", who, (long long)k64, KNN_MAX_K);
        return KNN_ERR_LIMIT;
    }
    if (nq > (int64_t(1) << 17)) {
        set_error("%s: at most 131072 queries per two-phase search (candidate lists stay resident)", who);
        return KNN_ERR_LIMIT;
    }
    const int k = int(k64);
    KNN_CHECK_CUDA(cudaStreamWaitEvent(s, ix->add_event, 0));
    ix->st_gemm_launches = 0;
    ix->st_gemm_ms = 0;
    ix->st_rerank_ms = 0;
    ix->ev_used_r = 0;
    ix->st_overflow_batches = 0;
    ix->st_overflow_queries = 0;
    ix->ev_used = 0;
    auto& P = ix->pend;
    P = knn_index::Pending();
    P.nq = nq;
    P.k = k;
    P.xq = xq_dev;
    P.dtype = qdt;
    P.launches0 = g_launches.load();
    P.tensor = ix->ntotal > 0 && use_tensor_path(ix, nq, k);
    ix->last_path = P.tensor ? 2 : 1;
    // The batch geometry depends on nq and query_batch alone, never on the path: the shards of one search lay out
    // their bound slots [batch][shard][2 * rows] from it and exchange bounds batch by batch, so a shard on the exact
    // path (fewer rows than tensor_min_n or than k, empty, path = 1) must cut the queries exactly as the others do.
    P.qb = round_up(std::min<int64_t>(ix->query_batch, nq), 256);
    P.nbatches = (nq + P.qb - 1) / P.qb;
    if (!P.tensor) {  // exact path: nothing to filter, no bound to offer; finish scans each batch's queries
        P.active = true;
        return KNN_OK;
    }
    KNN_CHECK(prepare_shadow(ix, k, s));
    P.cap = candidate_capacity(k, ix->ntotal, ix->dense_small_db != 0);
    KNN_CHECK(tensor_ws_ensure(ix->ws2, P.nbatches * P.qb, ix->dp, P.cap));
    KNN_CHECK(ix->overflow.ensure(sizeof(int) * size_t(P.nbatches)));
    KNN_CHECK(ix->ovf_q.ensure(sizeof(int) * size_t(nq)));
    KNN_CHECK(tensor_prepare(ix));
    KNN_CHECK_CUDA(cudaMemsetAsync(ix->overflow.p, 0, sizeof(int) * size_t(P.nbatches), s));
    P.active = true;
    return KNN_OK;
}

// Filter of batch b.  lower[q] = thr + eps = (k-th best approximate score) - eps, a lower bound of the true k-th best
// score of the shard; second bound (j >= 1): (j-th best approximate score) - eps - with G shards and j = ceil(k / G)
// the MIN of it over the shards is a lower bound of the global k-th best (every shard holds j rows at or above it).
// `negate_j`: the second bound is written negated, so that ONE element-wise MAX reduction combines both.
static int two_phase_filter_batch(knn_index* ix, int64_t b, float* lower_b, int64_t j, float* lower_j_b, bool negate_j,
                                  cudaStream_t s) {
    auto& P = ix->pend;
    const int64_t q0 = b * P.qb;
    const int64_t nb = P.nq - q0 < P.qb ? P.nq - q0 : P.qb;
    if (lower_j_b && (j < 1 || j > P.k)) {
        set_error("search_filter: j must be in [1, k]");
        return KNN_ERR_INVALID;
    }
    if (!P.tensor) {
        KNN_CHECK(launch_fill_f32(lower_b, nb, -FLT_MAX, s));
        if (lower_j_b) KNN_CHECK(launch_fill_f32(lower_j_b, nb, negate_j ? FLT_MAX : -FLT_MAX, s));
        return KNN_OK;
    }
    KNN_CHECK(tensor_filter_batch(ix, ix->ws2, q0, nb, row_at(P.xq, q0, ix->d, P.dtype), P.dtype, P.k, P.cap,
                                  ix->overflow.as<int>() + b, ix->ovf_q.as<int>() + q0, s));
    KNN_CHECK(launch_export_lower(ix->ws2.thr.as<float>() + q0, ix->ws2.eps.as<float>() + q0, nb, lower_b, s));
    if (lower_j_b) {
        KNN_CHECK(launch_kth_lower(filter_state(ix->ws2, q0, P.cap), ix->ws2.eps.as<float>() + q0, nb, int(j), negate_j, lower_j_b, s));
    }
    return KNN_OK;
}

static int two_phase_finish_batch(knn_index* ix, int64_t b, const float* lower_b, const float* neg_lower2_b, float* D_dev,
                                  int64_t* I_dev, int64_t id_base, cudaStream_t s) {
    auto& P = ix->pend;
    const int64_t q0 = b * P.qb;
    const int64_t nb = P.nq - q0 < P.qb ? P.nq - q0 : P.qb;
    if (!P.tensor) {
        // rows [q0, q0 + nb) by the exact scan (padding when the shard is empty).  A slice of the queries takes the exact
        // path whenever all of them do.  The scan uses the index's shared scratch (xq_f32, scores, lists): every batch of
        // an exact shard must be finished on the same stream.
        const long long l0 = P.launches0;
        KNN_CHECK(search_dev_impl(ix, nb, row_at(P.xq, q0, ix->d, P.dtype), P.dtype, P.k, D_dev + q0 * P.k, I_dev + q0 * P.k,
                                  id_base, s));
        P.launches0 = l0;
        return KNN_OK;
    }
    return tensor_finish_batch(ix, ix->ws2, q0, nb, P.k, P.cap, lower_b, neg_lower2_b, D_dev + q0 * P.k, I_dev + q0 * P.k, id_base, s);
}

static int two_phase_end(knn_index* ix, float* D_dev, int64_t* I_dev, int64_t id_base, cudaStream_t s) {
    auto& P = ix->pend;
    P.active = false;
    if (P.tensor) KNN_CHECK(redo_overflowed(ix, P.nq, P.qb, P.nbatches, P.xq, P.dtype, P.k, D_dev, I_dev, id_base, s));
    KNN_CHECK_CUDA(cudaEventRecord(ix->search_event, s));
    if (ix->profile && ix->ev_used) {
        KNN_CHECK_CUDA(cudaStreamSynchronize(s));
        collect_profile(ix);
    }
    ix->st_launches = g_launches.load() - P.launches0;
    return KNN_OK;
}

int knn_index_search_begin_typed_dev(knn_index* ix, int64_t nq, const void* xq_dev, int dtype, int64_t k,
                                     int64_t* nbatches_out, int64_t* batch_rows_out, void* stream) {
    if (!ix || !nbatches_out || !batch_rows_out) {
        set_error("search_begin: invalid arguments");
        return KNN_ERR_INVALID;
    }
    DeviceGuard g(ix->device);
    KNN_CHECK(two_phase_begin(ix, nq, xq_dev, dtype, k, static_cast<cudaStream_t>(stream), "search_begin"));
    *nbatches_out = ix->pend.nbatches;
    *batch_rows_out = ix->pend.qb;
    return KNN_OK;
}

int knn_index_search_begin_dev(knn_index* ix, int64_t nq, const float* xq_dev, int64_t k, int64_t* nbatches_out,
                               int64_t* batch_rows_out, void* stream) {
    return knn_index_search_begin_typed_dev(ix, nq, xq_dev, KNN_DTYPE_F32, k, nbatches_out, batch_rows_out, stream);
}

int knn_index_search_filter_batch_dev(knn_index* ix, int64_t b, int64_t j, float* bounds_dev, void* stream) {
    if (!ix || !bounds_dev || !ix->pend.active || b < 0 || b >= ix->pend.nbatches) {
        set_error("search_filter_batch: no search_begin pending, batch out of range or null bounds");
        return KNN_ERR_INVALID;
    }
    DeviceGuard g(ix->device);
    float* base = bounds_dev + b * 2 * ix->pend.qb;
    return two_phase_filter_batch(ix, b, base, j > 0 ? j : 1, base + ix->pend.qb, /*negate_j=*/true, static_cast<cudaStream_t>(stream));
}

int knn_index_search_finish_batch_dev(knn_index* ix, int64_t b, const float* bounds_dev, float* D_dev, int64_t* I_dev,
                                      int64_t id_base, void* stream) {
    if (!ix || !D_dev || !I_dev || !ix->pend.active || b < 0 || b >= ix->pend.nbatches) {
        set_error("search_finish_batch: no search_begin pending, batch out of range or null output");
        return KNN_ERR_INVALID;
    }
    DeviceGuard g(ix->device);
    const float* base = bounds_dev ? bounds_dev + b * 2 * ix->pend.qb : nullptr;
    return two_phase_finish_batch(ix, b, base, base ? base + ix->pend.qb : nullptr, D_dev, I_dev, id_base, static_cast<cudaStream_t>(stream));
}

int knn_index_search_end_dev(knn_index* ix, float* D_dev, int64_t* I_dev, int64_t id_base, void* stream) {
    if (!ix || !D_dev || !I_dev || !ix->pend.active) {
        set_error("search_end: no search_begin pending");
        return KNN_ERR_INVALID;
    }
    DeviceGuard g(ix->device);
    return two_phase_end(ix, D_dev, I_dev, id_base, static_cast<cudaStream_t>(stream));
}

int knn_index_search_filter_typed_dev(knn_index* ix, int64_t nq, const void* xq_dev, int dtype, int64_t k64, float* lower_dev,
                                      int64_t j, float* lower_j_dev, void* stream) {
    if (!ix || !lower_dev) {
        set_error("search_filter: invalid arguments");
        return KNN_ERR_INVALID;
    }
    DeviceGuard g(ix->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    KNN_CHECK(two_phase_begin(ix, nq, xq_dev, dtype, k64, s, "search_filter"));
    auto& P = ix->pend;
    for (int64_t b = 0; b < P.nbatches; ++b) {
        const int64_t q0 = b * P.qb;
        const int rc = two_phase_filter_batch(ix, b, lower_dev + q0, j, lower_j_dev ? lower_j_dev + q0 : nullptr, false, s);
        if (rc != KNN_OK) {
            P.active = false;
            return rc;
        }
    }
    return KNN_OK;
}

int knn_index_search_filter_dev(knn_index* ix, int64_t nq, const float* xq_dev, int64_t k64, float* lower_dev, int64_t j,
                                float* lower_j_dev, void* stream) {
    return knn_index_search_filter_typed_dev(ix, nq, xq_dev, KNN_DTYPE_F32, k64, lower_dev, j, lower_j_dev, stream);
}

int knn_index_search_finish_typed_dev(knn_index* ix, int64_t nq, const void* xq_dev, int dtype, int64_t k64,
                                      const float* lower_dev, float* D_dev, int64_t* I_dev, int64_t id_base, void* stream) {
    if (!ix || !xq_dev || !D_dev || !I_dev) {
        set_error("search_finish: invalid arguments");
        return KNN_ERR_INVALID;
    }
    KNN_CHECK(check_dtype(dtype, "search_finish"));
    auto& P = ix->pend;
    if (!P.active || P.nq != nq || P.k != int(k64) || P.xq != xq_dev || P.dtype != dtype) {
        set_error("search_finish: no matching search_filter call is pending");
        return KNN_ERR_INVALID;
    }
    DeviceGuard g(ix->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    for (int64_t b = 0; b < P.nbatches; ++b) {
        const int rc = two_phase_finish_batch(ix, b, lower_dev ? lower_dev + b * P.qb : nullptr, nullptr, D_dev, I_dev, id_base, s);
        if (rc != KNN_OK) {
            P.active = false;
            return rc;
        }
    }
    return two_phase_end(ix, D_dev, I_dev, id_base, s);
}

int knn_index_search_finish_dev(knn_index* ix, int64_t nq, const float* xq_dev, int64_t k64, const float* lower_dev,
                                float* D_dev, int64_t* I_dev, int64_t id_base, void* stream) {
    return knn_index_search_finish_typed_dev(ix, nq, xq_dev, KNN_DTYPE_F32, k64, lower_dev, D_dev, I_dev, id_base, stream);
}

int knn_index_reconstruct(knn_index* ix, int64_t i0, int64_t n, float* out) {
    if (!ix || i0 < 0 || n < 0 || i0 + n > ix->ntotal || (n > 0 && !out)) {
        set_error("reconstruct: invalid range");
        return KNN_ERR_INVALID;
    }
    if (n == 0) return KNN_OK;
    DeviceGuard g(ix->device);
    KNN_CHECK_CUDA(cudaStreamSynchronize(ix->stream));
    if (ix->xb_f32) {
        KNN_CHECK_CUDA(cudaMemcpy2D(out, size_t(ix->d) * sizeof(float), ix->xb_f32 + i0 * ix->dp, size_t(ix->dp) * sizeof(float),
                                    size_t(ix->d) * sizeof(float), size_t(n), cudaMemcpyDeviceToHost));
    } else {
        std::vector<uint16_t> tmp(size_t(n) * ix->d);
        KNN_CHECK_CUDA(cudaMemcpy2D(tmp.data(), size_t(ix->d) * 2, ix->xb_h16 + i0 * ix->dp, size_t(ix->dp) * 2,
                                    size_t(ix->d) * 2, size_t(n), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < tmp.size(); ++i) {
            uint32_t u = uint32_t(tmp[i]) << 16;
            memcpy(out + i, &u, 4);
        }
    }
    return KNN_OK;
}

int knn_merge_topk_dev(int metric, int64_t nq, int64_t k, int nlists, const float* D_lists_dev, const int64_t* I_lists_dev,
                       float* D_out_dev, int64_t* I_out_dev, void* stream) {
    if (nq < 0 || k <= 0 || nlists <= 0 || (nq > 0 && (!D_lists_dev || !I_lists_dev || !D_out_dev || !I_out_dev))) {
        set_error("merge: invalid arguments");
        return KNN_ERR_INVALID;
    }
    if (k > KNN_MAX_K) {
        set_error("merge: k=%lld exceeds KNN_MAX_K=%d", (long long)k, KNN_MAX_K);
        return KNN_ERR_LIMIT;
    }
    PtrDeviceGuard g(D_out_dev);
    return launch_merge_lists(D_lists_dev, I_lists_dev, nlists, nq, int(k), metric == KNN_METRIC_INNER_PRODUCT, D_out_dev,
                              I_out_dev, static_cast<cudaStream_t>(stream));
}

int knn_index_set_param(knn_index* ix, const char* name, int64_t value) {
    if (!ix || !name) return KNN_ERR_INVALID;
    std::string n(name);
    if (n == "path" && value >= 0 && value <= 2) ix->path_param = int(value);
    else if (n == "query_batch" && value >= 128) ix->query_batch = round_up(value, 256);
    else if (n == "profile") ix->profile = value != 0;
    else if (n == "cta_group" && (value == 1 || value == 2)) ix->cta_group = int(value);
    else if (n == "l2_hints") ix->l2_hints = value != 0;
    else if (n == "gemm_stages" && value >= 0 && value <= 6) ix->gemm_stages = int(value);
    else if (n == "stream_kernel") ix->stream_kernel = value != 0;
    else if (n == "overlap_finish") ix->overlap_finish = value != 0;
    else if (n == "small_m128") ix->small_m128 = value != 0;
    else if (n == "stream_pair") ix->stream_pair = value != 0;
    else if (n == "dense_small_db") ix->dense_small_db = value != 0;
    else if (n == "stream_quad") ix->stream_quad = value != 0;
    else if (n == "l2_blocked_rerank") ix->l2_blocked_rerank = value != 0;
    else if (n == "split_single_batch") ix->split_single_batch = value != 0;
    else if (n == "panel_ratio" && value >= 0 && value <= 64) ix->panel_ratio = int(value);
    else if (n == "small_batch_nq" && value >= 0) ix->small_batch_nq = value;
#ifdef KNN_EXPERIMENTS  // measurement aid that skips the epilogue (wrong results): never part of the shipped ABI
    else if (n == "debug_skip_epilogue") ix->debug_skip_epilogue = int(value);
#endif
    else if (n == "shadow_fmt" && value >= 0 && value <= 2) {  // takes effect at the next search (prepare_shadow)
        if (bf16_only(ix) && value == 2) {
            set_error("set_param: an index with bf16 storage keeps bf16 rows");
            return KNN_ERR_INVALID;
        }
        ix->shadow_param = int(value);
    }
    else if (n == "mantissa_bits" && (value == 0 || (value >= 2 && value <= 7))) ix->mbits_param = int(value);
    else if (n == "tensor_min_nq" && value >= 1) ix->tensor_min_nq = value;
    else if (n == "tensor_min_n" && value >= 1) ix->tensor_min_n = value;
    else {
        set_error("set_param: unknown parameter or bad value: %s=%lld", name, (long long)value);
        return KNN_ERR_INVALID;
    }
    return KNN_OK;
}

int knn_index_get_stat(const knn_index* ix, const char* name, double* out) {
    if (!ix || !name || !out) return KNN_ERR_INVALID;
    std::string n(name);
    if (n == "path") *out = ix->last_path;
    else if (n == "launches") *out = double(ix->st_launches);
    else if (n == "gemm_launches") *out = double(ix->st_gemm_launches);
    else if (n == "gemm_ms") *out = ix->st_gemm_ms;
    else if (n == "rerank_ms") *out = ix->st_rerank_ms;
    else if (n == "overflow_batches") *out = double(ix->st_overflow_batches);
    else if (n == "overflow_queries") *out = double(ix->st_overflow_queries);
    else if (n == "capacity") *out = double(ix->capacity);
    else if (n == "shadow_fmt") *out = ix->shadow_fmt == kFmtFP16 ? 2 : 1;
    else if (n == "mantissa_bits") *out = ix->shadow_fmt == kFmtFP16 ? 10 : ix->shadow_mbits;
    else if (n == "shadow_conversions") *out = double(ix->st_shadow_conversions);
    else {
        set_error("get_stat: unknown statistic %s", name);
        return KNN_ERR_INVALID;
    }
    return KNN_OK;
}

}  // extern "C"

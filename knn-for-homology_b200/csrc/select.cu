// Top-k selection kernels: radix narrowing on composite (score, id) keys followed by a
// shared-memory bitonic sort of the few survivors.  One CTA per (query, segment).
//
// Replaces the per-query heap / reservoir of faiss's result handlers (upstream faiss
// utils/Heap.h, ResultHandler.h - third-party, see oracle/flat_oracle.py) behind
// index.search (cath/search.py:24, pfam/proteins_search.py:49, seqvec_search/main.py:45):
// best first, equal scores -> lower id first, label -1 / +-FLT_MAX padding.
#include "common.cuh"

namespace knn {
namespace {

struct SelectSmem {
    uint64_t keys[kSortCap];
    int hist[256];
    uint64_t red_a[32];
    uint64_t red_b[32];
    int scount;
    int bucket;
    int cum_gt;
    int bucket_count;
};

// Narrow [prefix, mask] one 8-bit digit at a time (most significant differing bit first) until
// the boundary bucket plus everything strictly above it fits in `stop` elements, or all bits are
// fixed.  On return every key with (key & mask) > prefix is among the `k` best, `need` more have
// to come out of the bucket (key & mask) == prefix, which holds `bucket_count` keys.
template <typename Key, class Gen>
__device__ void radix_narrow(const Gen& gen, int L, int k, int stop, Key mn, Key mx, int* hist, int* sh_bucket,
                             int* sh_cum, int* sh_cnt, Key& prefix, Key& mask, int& need, int& bucket_count) {
    constexpr int kBits = int(sizeof(Key)) * 8;
    const int tid = threadIdx.x, T = blockDim.x;
    const Key diff = mn ^ mx;
    const int hi_bit = kBits - 1 - (sizeof(Key) == 8 ? __clzll((long long)diff) : __clz((int)diff));
    int shift = hi_bit >= 7 ? hi_bit - 7 : 0;
    mask = hi_bit == kBits - 1 ? Key(0) : Key(~Key(0)) << (hi_bit + 1);
    prefix = mx & mask;
    need = k;
    for (;;) {
        for (int i = tid; i < 256; i += T) hist[i] = 0;
        __syncthreads();
        for (int i = tid; i < L; i += T) {
            const Key key = gen(i);
            if ((key & mask) == prefix) atomicAdd(&hist[int((key >> shift) & Key(0xFF))], 1);
        }
        __syncthreads();
        if (tid < 32) {
            int loc[8];
            int s = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                loc[j] = hist[8 * tid + j];
                s += loc[j];
            }
            int suf = s;  // inclusive suffix sum over lanes (bins of this lane and all higher lanes)
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const int v = __shfl_down_sync(0xffffffffu, suf, off);
                if (tid + off < 32) suf += v;
            }
            const int above = suf - s;
            if (above < need && need <= above + s) {  // exactly one lane owns the boundary bucket
                int cum = above;
#pragma unroll
                for (int j = 7; j >= 0; --j) {
                    if (cum + loc[j] >= need) {
                        *sh_bucket = 8 * tid + j;
                        *sh_cum = cum;
                        *sh_cnt = loc[j];
                        break;
                    }
                    cum += loc[j];
                }
            }
        }
        __syncthreads();
        const int b = *sh_bucket;
        need -= *sh_cum;
        bucket_count = *sh_cnt;
        prefix |= Key(b) << shift;
        mask |= Key(0xFF) << shift;
        if ((k - need) + bucket_count <= stop || shift == 0) break;
        shift = shift >= 8 ? shift - 8 : 0;
    }
}

template <typename Key>
__device__ void block_minmax(Key mn, Key mx, Key* red_a, Key* red_b, Key& out_mn, Key& out_mx) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const Key a = __shfl_xor_sync(0xffffffffu, mn, off);
        const Key b = __shfl_xor_sync(0xffffffffu, mx, off);
        mn = a < mn ? a : mn;
        mx = b > mx ? b : mx;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    if (lane == 0) {
        red_a[warp] = mn;
        red_b[warp] = mx;
    }
    __syncthreads();
    mn = red_a[0];
    mx = red_b[0];
    for (int w = 1; w < nw; ++w) {
        mn = red_a[w] < mn ? red_a[w] : mn;
        mx = red_b[w] > mx ? red_b[w] : mx;
    }
    out_mn = mn;
    out_mx = mx;
    __syncthreads();
}

__device__ void bitonic_sort_desc(uint64_t* keys, int P) {
    const int tid = threadIdx.x, T = blockDim.x;
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = tid; i < (P >> 1); i += T) {
                const int pos = 2 * i - (i & (stride - 1));
                const int j = pos + stride;
                const uint64_t a = keys[pos], b = keys[j];
                const bool desc = (pos & size) == 0;
                if ((a < b) == desc) {
                    keys[pos] = b;
                    keys[j] = a;
                }
            }
        }
    }
    __syncthreads();
}

// Leaves the best min(k, L) keys of gen(0..L) sorted (descending) in sm.keys[0..) and returns
// their number.  Requires k <= kSortCap / 2.  Keys equal to 0 are padding and sort last.
template <class Gen>
__device__ int block_select_sorted(const Gen& gen, int L, int k, SelectSmem& sm) {
    const int tid = threadIdx.x, T = blockDim.x;
    int n;
    if (L <= kSortCap) {
        for (int i = tid; i < L; i += T) sm.keys[i] = gen(i);
        n = L;
    } else {
        uint64_t mn = ~0ull, mx = 0ull;
        for (int i = tid; i < L; i += T) {
            const uint64_t key = gen(i);
            mn = key < mn ? key : mn;
            mx = key > mx ? key : mx;
        }
        block_minmax<uint64_t>(mn, mx, sm.red_a, sm.red_b, mn, mx);
        if (mn == mx) {  // only possible when every key is padding
            n = k < L ? k : L;
            for (int i = tid; i < n; i += T) sm.keys[i] = mx;
        } else {
            uint64_t prefix, mask;
            int need, bucket_count;
            radix_narrow<uint64_t>(gen, L, k, kSortCap, mn, mx, sm.hist, &sm.bucket, &sm.cum_gt, &sm.bucket_count,
                                   prefix, mask, need, bucket_count);
            // First every key strictly above the boundary bucket (fewer than k <= kSortCap / 2 of them: none may be
            // lost), then the bucket's keys while there is room.  The bucket only exceeds the room when the narrowing
            // ran out of bits, i.e. its keys are identical - padding (valid keys are distinct) - so dropping some is
            // harmless; taking bucket keys in the same pass could crowd out real keys, e.g. a rescored list in which
            // fewer than k entries are still valid and thousands are padding.
            if (tid == 0) sm.scount = 0;
            __syncthreads();
            for (int i = tid; i < L; i += T) {
                const uint64_t key = gen(i);
                if ((key & mask) > prefix) {
                    const int p = atomicAdd(&sm.scount, 1);
                    if (p < kSortCap) sm.keys[p] = key;  // always true: fewer than k keys lie above the bucket
                }
            }
            __syncthreads();
            for (int i = tid; i < L; i += T) {
                const uint64_t key = gen(i);
                if ((key & mask) == prefix) {
                    const int p = atomicAdd(&sm.scount, 1);
                    if (p < kSortCap) sm.keys[p] = key;
                }
            }
            __syncthreads();
            n = sm.scount < kSortCap ? sm.scount : kSortCap;
        }
    }
    int P = 2;
    while (P < n) P <<= 1;
    for (int i = n + tid; i < P; i += T) sm.keys[i] = 0ull;
    bitonic_sort_desc(sm.keys, P);
    return n < k ? n : k;
}

// ---------------------------------------------------------------------------------------
// FILT: an ineligible row becomes the padding key 0 by its id (any score, -FLT_MAX and +FLT_MAX included, is one a row
// can really have), so it never enters a segment list.
template <bool FILT>
__global__ void __launch_bounds__(kSelectThreads)
select_dense_kernel(const float* __restrict__ scores, int64_t ld, int64_t ncols, int seg_len, uint32_t id_base, int k,
                    int largest, float* __restrict__ list_scores, uint32_t* __restrict__ list_ids, int64_t list_ld,
                    int64_t list_off, const RowFilter filt) {
    __shared__ SelectSmem sm;
    const int64_t q = blockIdx.y;
    const int64_t seg = blockIdx.x;
    const int64_t c0 = seg * seg_len;
    const int L = int((ncols - c0) < seg_len ? (ncols - c0) : seg_len);
    const float* row = scores + q * ld + c0;
    const uint32_t base = id_base + uint32_t(c0);
    int n;
    if constexpr (FILT) {
        const int64_t ex_row = excluded_row(filt, q);
        auto gen = [=] __device__(int i) {
            const uint32_t r = base + uint32_t(i);
            if (int64_t(r) == ex_row || !row_allowed(filt, r)) return uint64_t(0);
            return make_key(row[i], r, largest);
        };
        n = block_select_sorted(gen, L, k, sm);
    } else {
        auto gen = [=] __device__(int i) { return make_key(row[i], base + uint32_t(i), largest); };
        n = block_select_sorted(gen, L, k, sm);
    }
    float* os = list_scores + q * list_ld + list_off + seg * k;
    uint32_t* oi = list_ids + q * list_ld + list_off + seg * k;
    for (int r = threadIdx.x; r < k; r += blockDim.x) {
        const uint64_t key = r < n ? sm.keys[r] : 0ull;
        os[r] = key ? key_score(key, largest) : 0.f;
        oi[r] = key ? key_id(key) : kInvalidId;
    }
}

__device__ __forceinline__ void write_final(const SelectSmem& sm, int n, int k, int largest, float* D, int64_t* I,
                                            int64_t id_base) {
    for (int r = threadIdx.x; r < k; r += blockDim.x) {
        const uint64_t key = r < n ? sm.keys[r] : 0ull;
        if (key) {
            D[r] = key_score(key, largest);
            I[r] = int64_t(key_id(key)) + id_base;
        } else {  // heap neutral element of faiss: label -1
            D[r] = largest ? -FLT_MAX : FLT_MAX;
            I[r] = -1;
        }
    }
}

__global__ void __launch_bounds__(kSelectThreads)
select_final_kernel(const float* __restrict__ list_scores, const uint32_t* __restrict__ list_ids,
                    const int* __restrict__ counts, int64_t list_ld, int64_t fixed_len, int k, int largest,
                    float* __restrict__ D, int64_t* __restrict__ I, int64_t id_base) {
    __shared__ SelectSmem sm;
    const int64_t q = blockIdx.x;
    int64_t len = fixed_len;
    if (counts) len = counts[q] < list_ld ? counts[q] : list_ld;
    const float* ls = list_scores + q * list_ld;
    const uint32_t* li = list_ids + q * list_ld;
    auto gen = [=] __device__(int i) { return make_key(ls[i], li[i], largest); };
    const int n = block_select_sorted(gen, int(len), k, sm);
    write_final(sm, n, k, largest, D + q * k, I + q * k, id_base);
}

__global__ void __launch_bounds__(kSelectThreads)
merge_lists_kernel(const float* __restrict__ D_lists, const int64_t* __restrict__ I_lists, int nlists, int64_t nq,
                   int k, int largest, float* __restrict__ D, int64_t* __restrict__ I) {
    __shared__ SelectSmem sm;
    const int64_t q = blockIdx.x;
    auto gen = [=] __device__(int i) {
        const int l = i / k, r = i - l * k;
        const int64_t off = (int64_t(l) * nq + q) * k + r;
        const int64_t id = I_lists[off];
        return make_key(D_lists[off], id < 0 ? kInvalidId : uint32_t(id), largest);
    };
    const int n = block_select_sorted(gen, nlists * k, k, sm);
    write_final(sm, n, k, largest, D + q * k, I + q * k, 0);
}

// ---------------------------------------------------------------------------------------
// Tighten: per query, k-th best approximate score so far -> new candidate threshold, then drop
// the candidates that fell below it (order-preserving in-place compaction).
struct TightenSmem {
    int hist[256];
    uint32_t red_a[32];
    uint32_t red_b[32];
    int bucket;
    int cum_gt;
    int bucket_count;
    int warp_tot[32];
    int base;
};

__global__ void __launch_bounds__(256)
tighten_kernel(float* __restrict__ thr, int* __restrict__ counts, float* __restrict__ cand_scores,
               uint32_t* __restrict__ cand_ids, int cap, const float* __restrict__ eps, int k, int compact,
               int* __restrict__ overflow, int* __restrict__ ovf_q) {
    __shared__ TightenSmem sm;
    const int64_t q = blockIdx.x;
    const int tid = threadIdx.x, T = blockDim.x;
    int cnt = counts[q];
    if (cnt > cap) {
        if (tid == 0) {
            atomicExch(overflow, 1);
            ovf_q[q] = 1;
        }
        cnt = cap;
    }
    if (cnt < k || cnt == 0) return;  // fewer than k candidates seen: everything stays a candidate
    float* cs = cand_scores + q * int64_t(cap);
    uint32_t* ci = cand_ids + q * int64_t(cap);
    // (Staging the list in shared memory as keys so that the radix passes run on-chip was measured: 5.6 vs 5.2 ms for
    // the 14 launches of two C3 batches - the 32 KB per CTA cost more occupancy than the L2-resident re-reads cost time.)
    auto gen = [=] __device__(int i) {
        const float s = cs[i];
        return s != s ? 0u : orderable_f32(s);
    };
    uint32_t mn = ~0u, mx = 0u;
    for (int i = tid; i < cnt; i += T) {
        const uint32_t key = gen(i);
        mn = key < mn ? key : mn;
        mx = key > mx ? key : mx;
    }
    block_minmax<uint32_t>(mn, mx, sm.red_a, sm.red_b, mn, mx);
    uint32_t kth = mx;
    if (mn != mx) {
        uint32_t prefix, mask;
        int need, bucket_count;
        radix_narrow<uint32_t>(gen, cnt, k, 0, mn, mx, sm.hist, &sm.bucket, &sm.cum_gt, &sm.bucket_count, prefix, mask,
                               need, bucket_count);
        kth = prefix;  // all bits fixed: the k-th largest key itself
    }
    const float kth_score = from_orderable_f32(kth);
    const float e = eps[q];
    float t = kth_score - 2.0f * e;
    if (!(t == t)) t = -FLT_MAX;
    // the bound only ever rises (k-th best over a superset); keep the max for safety with NaNs
    const float old = thr[q];
    if (old > t) t = old;
    __syncthreads();
    if (tid == 0) thr[q] = t;
    if (!compact) return;
    // ordered compaction, chunk by chunk: writes land at or before the positions already read
    if (tid == 0) sm.base = 0;
    __syncthreads();
    const int lane = tid & 31, warp = tid >> 5, nw = T >> 5;
    for (int c0 = 0; c0 < cnt; c0 += T) {
        const int i = c0 + tid;
        float s = 0.f;
        uint32_t id = kInvalidId;
        bool keep = false;
        if (i < cnt) {
            s = cs[i];
            id = ci[i];
            keep = (s >= t) && id != kInvalidId;
        }
        const unsigned ballot = __ballot_sync(0xffffffffu, keep);
        const int wpre = __popc(ballot & ((1u << lane) - 1u));
        if (lane == 0) sm.warp_tot[warp] = __popc(ballot);
        __syncthreads();  // all reads of this chunk done, warp totals visible
        int off = sm.base;
        for (int w = 0; w < warp; ++w) off += sm.warp_tot[w];
        if (keep) {
            cs[off + wpre] = s;
            ci[off + wpre] = id;
        }
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < nw; ++w) tot += sm.warp_tot[w];
            sm.base += tot;
        }
        __syncthreads();
    }
    if (tid == 0) counts[q] = sm.base;
}


// Warp-per-query variant for small k (candidate lists of a few hundred entries).  The whole list is
// loaded into registers with independent loads (one memory round trip), the k-th largest key is found by a
// bit-by-bit search (32 rounds of compare + warp reduce), and the survivors are written back compacted - no
// block-wide barriers, no dependent global loads, 8 queries per CTA.
// Lowest key bit worth resolving when a value resolution of `res` (> 0) is enough.  Orderable keys are spaced one
// float ulp apart and the ulp grows with the magnitude, so a key distance of 2^bit spans at most 2^bit ulps of the
// LARGEST magnitude in the band [mn, mx]: every bit below the returned one resolves less than `res` anywhere in it.
// (Whatever is returned, clearing low bits of the k-th largest key only lowers it: the bound stays valid.)
__device__ __forceinline__ int key_resolution_bit(uint32_t mn, uint32_t mx, float res) {
    if (!(res > 0.f) || mn > mx) return 0;
    const float m = fmaxf(fabsf(from_orderable_f32(mn)), fabsf(from_orderable_f32(mx)));
    if (!(m > 0.f) || !(m < FLT_MAX)) return 0;
    int ex;
    frexpf(m, &ex);                                    // m = f * 2^ex, f in [0.5, 1): ulp(m) = 2^(ex - 24)
    const float keys_in_res = ldexpf(res, 24 - ex);    // res / ulp(m)
    if (!(keys_in_res >= 2.f)) return 0;
    int bit = 0;
    while (bit < 30 && ldexpf(1.f, bit + 1) <= keys_in_res) ++bit;  // 2^bit <= keys_in_res
    return bit;
}

template <int MAXE>
__device__ __forceinline__ void warp_tighten_reg(float* __restrict__ cs, uint32_t* __restrict__ ci, int cnt, int k,
                                                 float two_eps, float old_thr, int lane, float& thr_out, int& cnt_out) {
    uint32_t keys[MAXE];
    uint32_t ids[MAXE];
#pragma unroll
    for (int e = 0; e < MAXE; ++e) {
        const int i = e * 32 + lane;
        const float sc = i < cnt ? cs[i] : 0.f;
        ids[e] = i < cnt ? ci[i] : kInvalidId;
        keys[e] = (i < cnt && sc == sc) ? orderable_f32(sc) : 0u;
    }
    // Bit-by-bit search of the k-th largest key, on the bits that matter only: the bits all keys share are skipped
    // (scores of one list live in a narrow band), and the search stops at a resolution of eps / 16 - the prefix found
    // so far with the remaining bits cleared is a LOWER bound of the k-th largest key, which is all the threshold
    // needs (it costs ~3 % more candidates and a third of the rounds).
    uint32_t mn = ~0u, mx = 0u;
    int nvalid = 0;
#pragma unroll
    for (int e = 0; e < MAXE; ++e) {
        if (keys[e]) {  // 0 = padding / NaN
            mn = keys[e] < mn ? keys[e] : mn;
            mx = keys[e] > mx ? keys[e] : mx;
            ++nvalid;
        }
    }
    mn = __reduce_min_sync(0xffffffffu, mn);
    mx = __reduce_max_sync(0xffffffffu, mx);
    nvalid = __reduce_add_sync(0xffffffffu, nvalid);
    int top = -1, low = 0;
    uint32_t kth = 0;                     // fewer than k real scores: no bound (the original all-bits search ends at 0)
    if (nvalid >= k) {
        top = mn < mx ? 31 - __clz(int(mn ^ mx)) : -1;            // highest bit in which two keys differ
        low = key_resolution_bit(mn, mx, two_eps * 0.03125f);     // bits below it resolve less than eps / 16
        kth = top < 0 ? mx : (top >= 31 ? 0u : (mx & ~((2u << top) - 1u)));  // the prefix every key shares
    }
#pragma unroll 1
    for (int bit = top; bit >= low; --bit) {
        const uint32_t cand = kth | (1u << bit);
        int c = 0;
#pragma unroll
        for (int e = 0; e < MAXE; ++e) c += keys[e] >= cand ? 1 : 0;
        c = __reduce_add_sync(0xffffffffu, c);
        if (c >= k) kth = cand;  // at least k keys are >= cand: the k-th largest starts with these bits
    }
    float t = from_orderable_f32(kth) - two_eps;
    if (!(t == t)) t = -FLT_MAX;
    if (old_thr > t) t = old_thr;
    int base = 0;
#pragma unroll
    for (int e = 0; e < MAXE; ++e) {
        if (e * 32 < cnt) {  // warp-uniform
            const float sc = from_orderable_f32(keys[e]);
            const bool keep = (sc >= t) && ids[e] != kInvalidId;
            const unsigned ballot = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                const int p = base + __popc(ballot & ((1u << lane) - 1u));
                cs[p] = sc;
                ci[p] = ids[e];
            }
            base += __popc(ballot);
        }
    }
    thr_out = t;
    cnt_out = base;
}

__device__ __forceinline__ uint32_t warp_kth_largest_mem(const float* __restrict__ cs, int cnt, int k, int lane) {
    uint32_t t = 0;
#pragma unroll 1
    for (int bit = 31; bit >= 0; --bit) {
        const uint32_t cand = t | (1u << bit);
        int c = 0;
        for (int i = lane; i < cnt; i += 32) {
            const float s = cs[i];
            c += (s == s && orderable_f32(s) >= cand) ? 1 : 0;
        }
        c = __reduce_add_sync(0xffffffffu, c);
        if (c >= k) t = cand;
    }
    return t;
}

__global__ void __launch_bounds__(256)
tighten_warp_kernel(float* __restrict__ thr, int* __restrict__ counts, float* __restrict__ cand_scores,
                    uint32_t* __restrict__ cand_ids, int cap, const float* __restrict__ eps, int64_t nq, int k,
                    int* __restrict__ overflow, int* __restrict__ ovf_q) {
    const int lane = threadIdx.x & 31;
    const int64_t q = int64_t(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (q >= nq) return;
    int cnt = counts[q];
    const float two_eps = 2.0f * eps[q];
    const float old = thr[q];
    if (cnt > cap) {
        if (lane == 0) {
            atomicExch(overflow, 1);
            ovf_q[q] = 1;
        }
        cnt = cap;
    }
    if (cnt < k || cnt == 0) return;  // fewer than k candidates seen: everything stays a candidate
    float* cs = cand_scores + q * int64_t(cap);
    uint32_t* ci = cand_ids + q * int64_t(cap);
    float t;
    int base;
    if (cnt <= 8 * 32) {
        warp_tighten_reg<8>(cs, ci, cnt, k, two_eps, old, lane, t, base);
    } else if (cnt <= 16 * 32) {
        warp_tighten_reg<16>(cs, ci, cnt, k, two_eps, old, lane, t, base);
    } else if (cnt <= 32 * 32) {
        warp_tighten_reg<32>(cs, ci, cnt, k, two_eps, old, lane, t, base);
    } else {
        const uint32_t kth = warp_kth_largest_mem(cs, cnt, k, lane);
        t = from_orderable_f32(kth) - two_eps;
        if (!(t == t)) t = -FLT_MAX;
        if (old > t) t = old;
        // ordered in-place compaction, 32 entries at a time (a chunk is read completely before it is written,
        // and writes land at or before positions that were already read)
        base = 0;
        for (int c0 = 0; c0 < cnt; c0 += 32) {
            const int i = c0 + lane;
            float s = 0.f;
            uint32_t id = kInvalidId;
            bool keep = false;
            if (i < cnt) {
                s = cs[i];
                id = ci[i];
                keep = (s >= t) && id != kInvalidId;
            }
            const unsigned ballot = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                const int p = base + __popc(ballot & ((1u << lane) - 1u));
                cs[p] = s;
                ci[p] = id;
            }
            base += __popc(ballot);
            __syncwarp();
        }
    }
    if (lane == 0) {
        thr[q] = t;
        counts[q] = base;
    }
}

// lower_j[q] = (j-th best approximate score of the list) - eps[q]: at least j rows of this shard have a TRUE
// score >= lower_j[q].  One warp per query; -FLT_MAX when the list holds fewer than j entries.
__global__ void __launch_bounds__(256)
kth_lower_kernel(const float* __restrict__ cand_scores, const int* __restrict__ counts, int cap,
                 const float* __restrict__ eps, int64_t nq, int j, int negate, float* __restrict__ lower_j) {
    const int lane = threadIdx.x & 31;
    const int64_t q = int64_t(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (q >= nq) return;
    int cnt = counts[q];
    cnt = cnt < cap ? cnt : cap;
    float out = -FLT_MAX;
    const float e = eps[q];
    if (cnt >= j && j > 0 && e < FLT_MAX) {
        const uint32_t kth = warp_kth_largest_mem(cand_scores + q * int64_t(cap), cnt, j, lane);
        out = from_orderable_f32(kth) - e;
        if (!(out == out)) out = -FLT_MAX;
    }
    if (lane == 0) lower_j[q] = negate ? -out : out;
}

// k-way merge of up to 32 SORTED lists by one warp per query: lane l owns list l and its head; every round the
// warp takes the best head (64-bit composite keys are distinct, so there are no ties), the owner advances.
__device__ __forceinline__ uint64_t warp_max_u64(uint64_t v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const uint64_t o = __shfl_xor_sync(0xffffffffu, v, off);
        v = o > v ? o : v;
    }
    return v;
}

__global__ void __launch_bounds__(256)
merge_sorted_lists_kernel(const float* __restrict__ D_lists, const int64_t* __restrict__ I_lists, int nlists, int64_t nq,
                          int k, int largest, float* __restrict__ D, int64_t* __restrict__ I) {
    const int lane = threadIdx.x & 31;
    const int64_t q = int64_t(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (q >= nq) return;
    const int64_t base = lane < nlists ? (int64_t(lane) * nq + q) * k : 0;
    int pos = 0;
    auto load_key = [&](int p) -> uint64_t {
        if (lane >= nlists || p >= k) return 0ull;
        const int64_t id = I_lists[base + p];
        return make_key(D_lists[base + p], id < 0 ? kInvalidId : uint32_t(id), largest);
    };
    uint64_t head = load_key(0);
    uint64_t next = load_key(1);  // one element of look-ahead hides most of the dependent-load latency
    for (int r = 0; r < k; ++r) {
        const uint64_t best = warp_max_u64(head);
        if (lane == 0) {
            if (best) {
                D[q * k + r] = key_score(best, largest);
                I[q * k + r] = int64_t(key_id(best));
            } else {
                D[q * k + r] = largest ? -FLT_MAX : FLT_MAX;
                I[q * k + r] = -1;
            }
        }
        if (best && head == best) {  // exactly one lane
            ++pos;
            head = next;
            next = load_key(pos + 1);
        }
    }
}

__global__ void export_lower_kernel(const float* __restrict__ thr, const float* __restrict__ eps, int64_t nq,
                                    float* __restrict__ lower) {
    const int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const float t = thr[q], e = eps[q];
    lower[q] = (t <= -FLT_MAX || !(e < FLT_MAX)) ? -FLT_MAX : t + e;
}

__global__ void apply_lower_kernel(float* __restrict__ thr, const float* __restrict__ eps, const float* __restrict__ lower,
                                   const float* __restrict__ neg_lower2, int64_t nq) {
    const int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    float l = lower[q];
    const float e = eps[q];
    if (neg_lower2) {  // the caller's bound is max(lower, -neg_lower2)
        const float l2 = -neg_lower2[q];
        if (l2 > l) l = l2;
    }
    if (l > -FLT_MAX && e < FLT_MAX) {
        const float t = l - e;
        if (t > thr[q]) thr[q] = t;
    }
}

__global__ void fill_f32_kernel(float* p, int64_t n, float v) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

__global__ void init_filter_kernel(float* thr, int* counts, int* ovf, int64_t nq, int64_t nq_pad, int first_count) {
    const int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (q >= nq_pad) return;
    thr[q] = q < nq ? -FLT_MAX : FLT_MAX;
    counts[q] = q < nq ? first_count : 0;
    if (q < nq) ovf[q] = 0;
}

// SRC: element type of the query rows (float, __half, __nv_bfloat16); the fp32 rows written are exact up-conversions.
__device__ __forceinline__ float elem_f32(float v) { return v; }
__device__ __forceinline__ float elem_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float elem_f32(__nv_bfloat16 v) { return __bfloat162float(v); }

template <class SRC>
__global__ void gather_rows_kernel(const SRC* __restrict__ xq, int d, const int* __restrict__ idx, float* __restrict__ out) {
    const SRC* src = xq + int64_t(idx[blockIdx.x]) * d;
    float* dst = out + int64_t(blockIdx.x) * d;
    for (int i = threadIdx.x; i < d; i += blockDim.x) dst[i] = elem_f32(src[i]);
}

__global__ void gather_ids_kernel(const int64_t* __restrict__ ids, const int* __restrict__ idx, int64_t n, int64_t* __restrict__ out) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) out[i] = ids[idx[i]];
}

__global__ void scatter_results_kernel(const float* __restrict__ Dt, const int64_t* __restrict__ It, const int* __restrict__ idx,
                                       int k, float* __restrict__ D, int64_t* __restrict__ I) {
    const int64_t q = idx[blockIdx.x];
    for (int r = threadIdx.x; r < k; r += blockDim.x) {
        D[q * k + r] = Dt[int64_t(blockIdx.x) * k + r];
        I[q * k + r] = It[int64_t(blockIdx.x) * k + r];
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------
int launch_select_dense(const float* scores, int64_t ld, int64_t ncols, int64_t nq, int seg_len, uint32_t id_base,
                        int k, int largest, float* list_scores, uint32_t* list_ids, int64_t list_ld,
                        int64_t list_off, const RowFilter& filt, cudaStream_t s) {
    if (nq <= 0 || ncols <= 0) return KNN_OK;
    const int64_t nseg = (ncols + seg_len - 1) / seg_len;
    for (int64_t q0 = 0; q0 < nq; q0 += 65535) {
        const int64_t qn = nq - q0 < 65535 ? nq - q0 : 65535;
        dim3 grid((unsigned)nseg, (unsigned)qn, 1u);
        if (filt.active())
            select_dense_kernel<true><<<grid, kSelectThreads, 0, s>>>(scores + q0 * ld, ld, ncols, seg_len, id_base, k, largest,
                                                                      list_scores + q0 * list_ld, list_ids + q0 * list_ld,
                                                                      list_ld, list_off, filt.queries_from(q0));
        else
            select_dense_kernel<false><<<grid, kSelectThreads, 0, s>>>(scores + q0 * ld, ld, ncols, seg_len, id_base, k, largest,
                                                                       list_scores + q0 * list_ld, list_ids + q0 * list_ld,
                                                                       list_ld, list_off, filt);
        KNN_CHECK_LAUNCH();
    }
    return KNN_OK;
}

int launch_select_final(const float* list_scores, const uint32_t* list_ids, const int* counts, int64_t list_ld,
                        int64_t fixed_len, int64_t nq, int k, int largest, float* D, int64_t* I, int64_t id_base,
                        cudaStream_t s) {
    if (nq <= 0) return KNN_OK;
    select_final_kernel<<<unsigned(nq), kSelectThreads, 0, s>>>(list_scores, list_ids, counts, list_ld, fixed_len, k,
                                                                largest, D, I, id_base);
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

int launch_merge_lists(const float* D_lists, const int64_t* I_lists, int nlists, int64_t nq, int k, int largest,
                       float* D, int64_t* I, cudaStream_t s) {
    if (nq <= 0) return KNN_OK;
    if (nlists <= 32) {  // the inputs are sorted search results: warp tournament instead of a full sort
        merge_sorted_lists_kernel<<<unsigned((nq + 7) / 8), 256, 0, s>>>(D_lists, I_lists, nlists, nq, k, largest, D, I);
        KNN_CHECK_LAUNCH();
        return KNN_OK;
    }
    merge_lists_kernel<<<unsigned(nq), kSelectThreads, 0, s>>>(D_lists, I_lists, nlists, nq, k, largest, D, I);
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

int launch_tighten(FilterState st, const float* eps, int64_t nq, int k, int compact, float* tau_out, int* overflow,
                   cudaStream_t s) {
    (void)tau_out;
    if (nq <= 0) return KNN_OK;
    // One warp per query needs thousands of queries to fill the GPU; a small batch (<= 512 queries) is latency-bound in
    // its bit-by-bit search, so it takes the block-per-query kernel (radix passes by 256 threads) whatever k is.
    if (k <= 256 && compact && nq > 512) {
        tighten_warp_kernel<<<unsigned((nq + 7) / 8), 256, 0, s>>>(st.thr, st.counts, st.cand_scores, st.cand_ids, st.cap,
                                                                   eps, nq, k, overflow, st.ovf);
    } else {
        tighten_kernel<<<unsigned(nq), 256, 0, s>>>(st.thr, st.counts, st.cand_scores, st.cand_ids, st.cap, eps, k,
                                                    compact, overflow, st.ovf);
    }
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

int launch_export_lower(const float* thr, const float* eps, int64_t nq, float* lower, cudaStream_t s) {
    export_lower_kernel<<<unsigned((nq + 255) / 256), 256, 0, s>>>(thr, eps, nq, lower);
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

int launch_kth_lower(FilterState st, const float* eps, int64_t nq, int j, bool negate, float* lower_j, cudaStream_t s) {
    kth_lower_kernel<<<unsigned((nq + 7) / 8), 256, 0, s>>>(st.cand_scores, st.counts, st.cap, eps, nq, j, negate ? 1 : 0, lower_j);
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

int launch_apply_lower(float* thr, const float* eps, const float* lower, const float* neg_lower2, int64_t nq, cudaStream_t s) {
    apply_lower_kernel<<<unsigned((nq + 255) / 256), 256, 0, s>>>(thr, eps, lower, neg_lower2, nq);
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

int launch_fill_f32(float* p, int64_t n, float v, cudaStream_t s) {
    fill_f32_kernel<<<unsigned((n + 255) / 256), 256, 0, s>>>(p, n, v);
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

int launch_init_filter(FilterState st, int64_t nq, int64_t nq_pad, int first_count, cudaStream_t s) {
    init_filter_kernel<<<unsigned((nq_pad + 255) / 256), 256, 0, s>>>(st.thr, st.counts, st.ovf, nq, nq_pad, first_count);
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

int launch_gather_rows(const void* xq, int xq_dtype, int d, const int* idx, int64_t n, float* out, cudaStream_t s) {
    if (n <= 0) return KNN_OK;
    switch (xq_dtype) {
        case KNN_DTYPE_F32: gather_rows_kernel<<<unsigned(n), 256, 0, s>>>(static_cast<const float*>(xq), d, idx, out); break;
        case KNN_DTYPE_F16: gather_rows_kernel<<<unsigned(n), 256, 0, s>>>(static_cast<const __half*>(xq), d, idx, out); break;
        case KNN_DTYPE_BF16:
            gather_rows_kernel<<<unsigned(n), 256, 0, s>>>(static_cast<const __nv_bfloat16*>(xq), d, idx, out);
            break;
        default:
            set_error("unknown query dtype %d", xq_dtype);
            return KNN_ERR_INVALID;
    }
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

int launch_gather_ids(const int64_t* ids, const int* idx, int64_t n, int64_t* out, cudaStream_t s) {
    if (n <= 0) return KNN_OK;
    gather_ids_kernel<<<unsigned((n + 255) / 256), 256, 0, s>>>(ids, idx, n, out);
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

int launch_scatter_results(const float* Dt, const int64_t* It, const int* idx, int64_t n, int k, float* D, int64_t* I,
                           cudaStream_t s) {
    if (n <= 0) return KNN_OK;
    scatter_results_kernel<<<unsigned(n), 256, 0, s>>>(Dt, It, idx, k, D, I);
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

}  // namespace knn

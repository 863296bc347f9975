// CUDA-core kernels of the flat-search path: row normalisation, database ingest (fp32 master +
// bf16 shadow + norms), query preparation, the exact fp32 scan and the exact fp32 rerank.
// All of them are HBM-bound streaming kernels: one warp per row, 16-byte loads, grid sized
// in multiples of the SM count.
//
// Reference semantics restated (no reference source exists for them: the arithmetic lives in
// faiss-cpu 1.7.2, see oracle/flat_oracle.py):
//   normalize_l2_kernel  <- faiss.normalize_L2        (cath/search.py:19, seqvec_search/main.py:31,34)
//   ingest_rows_kernel   <- IndexFlat.add             (cath/search.py:22, pfam/proteins_search.py:37)
//   scan_f32_kernel      <- IndexFlat.search, fp32    (cath/search.py:24, seqvec_search/main.py:45)
#include <algorithm>

#include "common.cuh"

namespace knn {

namespace {

constexpr int kWarpsPerBlock = 8;
constexpr int kBlock = kWarpsPerBlock * 32;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

int grid_for_rows(int64_t rows, int rows_per_block, int blocks_per_sm) {
    int64_t want = (rows + rows_per_block - 1) / rows_per_block;
    int64_t cap = int64_t(num_sms()) * blocks_per_sm;
    if (want < 1) want = 1;
    return int(want < cap ? want : cap);
}

// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) normalize_l2_kernel(float* __restrict__ x, int64_t n, int64_t d,
                                                               int vec_ok) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = int64_t(gridDim.x) * kWarpsPerBlock;
    for (int64_t row = int64_t(blockIdx.x) * kWarpsPerBlock + (threadIdx.x >> 5); row < n; row += warps) {
        float* r = x + row * d;
        float s = 0.f;
        if (vec_ok) {
            const float4* r4 = reinterpret_cast<const float4*>(r);
            for (int64_t c = lane; c < d / 4; c += 32) {
                float4 v = r4[c];
                s = fmaf(v.x, v.x, s); s = fmaf(v.y, v.y, s); s = fmaf(v.z, v.z, s); s = fmaf(v.w, v.w, s);
            }
        } else {
            for (int64_t c = lane; c < d; c += 32) s = fmaf(r[c], r[c], s);
        }
        s = warp_sum(s);
        if (s > 0.f) {
            const float inv = 1.0f / sqrtf(s);
            if (vec_ok) {
                float4* r4 = reinterpret_cast<float4*>(r);
                for (int64_t c = lane; c < d / 4; c += 32) {
                    float4 v = r4[c];
                    v.x *= inv; v.y *= inv; v.z *= inv; v.w *= inv;
                    r4[c] = v;
                }
            } else {
                for (int64_t c = lane; c < d; c += 32) r[c] *= inv;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// Rounds v (to nearest, ties to even) to `mbits` explicit mantissa bits; NaN / Inf pass through.
__device__ __forceinline__ float round_mantissa(float v, int mbits) {
    uint32_t u = __float_as_uint(v);
    if ((u & 0x7F800000u) == 0x7F800000u) return v;
    const int drop = 23 - mbits;
    u += ((1u << (drop - 1)) - 1u) + ((u >> drop) & 1u);
    u &= ~((1u << drop) - 1u);
    return __uint_as_float(u);
}

// fp32 pair -> packed 16-bit shadow pair + the values the shadow holds.
// bf16: `mbits` < 7 keeps fewer mantissa bits than the format has (see ShadowFmt in common.cuh: operand bits that
// never toggle cost no multiplier power, and the kernel is power-bound).
// fp16: finite values beyond the format's range saturate, values below its normal range flush to zero (no
// subnormal ever reaches the tensor cores).  Either way the loss shows up in |y - shadow(y)|, which is measured,
// never assumed.  NaN and Inf pass through unchanged: such a row never enters a result.
template <int FMT>
__device__ __forceinline__ uint32_t pack_shadow2(float a, float b, int mbits, float2& back) {
    if (FMT == kFmtFP16) {
        const float fa = fabsf(a), fb = fabsf(b);
        if (fa > 65504.f && fa <= FLT_MAX) a = copysignf(65504.f, a);
        if (fb > 65504.f && fb <= FLT_MAX) b = copysignf(65504.f, b);
        if (fa < 6.103515625e-05f) a = 0.f;
        if (fb < 6.103515625e-05f) b = 0.f;
        __half2 h = __floats2half2_rn(a, b);
        back = __half22float2(h);
        return *reinterpret_cast<uint32_t*>(&h);
    } else {
        if (mbits < 7) {
            a = round_mantissa(a, mbits);
            b = round_mantissa(b, mbits);
        }
        __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
        back = __bfloat1622float2(h);
        return *reinterpret_cast<uint32_t*>(&h);
    }
}

// Elements 4c .. 4c+3 of a caller row, converted to fp32 at the load.  fp16 -> fp32 and bf16 -> fp32 are exact, so
// everything downstream of the load sees exactly the values of the up-converted row.  16-bit sources load 8 bytes per
// 4 elements (a uint2, as RowChunk<true> below); the caller guarantees 16-byte (fp32) / 8-byte (16-bit) alignment.
__device__ __forceinline__ float4 load4_f32(const float* r, int c) { return reinterpret_cast<const float4*>(r)[c]; }
__device__ __forceinline__ float4 load4_f32(const __half* r, int c) {
    uint2 p = reinterpret_cast<const uint2*>(r)[c];
    const float2 a = __half22float2(*reinterpret_cast<__half2*>(&p.x));
    const float2 b = __half22float2(*reinterpret_cast<__half2*>(&p.y));
    return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float4 load4_f32(const __nv_bfloat16* r, int c) {
    const uint2 p = reinterpret_cast<const uint2*>(r)[c];  // bf16 -> fp32 is a 16-bit shift
    return make_float4(__uint_as_float(p.x << 16), __uint_as_float(p.x & 0xFFFF0000u), __uint_as_float(p.y << 16),
                       __uint_as_float(p.y & 0xFFFF0000u));
}
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }

// One warp per row.  Writes the zero-padded fp32 master row (optional), the 16-bit shadow row,
// |y|^2 and folds max|y|^2, max|y - shadow(y)|^2 into *stats (optional).
// SRC: element type of the caller's rows (float, __half or __nv_bfloat16); 16-bit rows run the fp32 arithmetic on
// their exact fp32 values, so every output is bit-identical to ingesting the up-converted rows.
template <int FMT, class SRC>
__global__ void __launch_bounds__(kBlock) ingest_rows_kernel(const SRC* __restrict__ src, int64_t src_ld, int64_t n,
                                                              int d, int dp, float* __restrict__ dst_f32,
                                                              h16_t* __restrict__ dst_h16,
                                                              float* __restrict__ norms2,
                                                              float* __restrict__ dnorms2, DbStats* stats,
                                                              int vec_ok, int shadow_is_master, int mbits) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = int64_t(gridDim.x) * kWarpsPerBlock;
    float wmax_n = 0.f, wmax_d = 0.f;
    for (int64_t row = int64_t(blockIdx.x) * kWarpsPerBlock + (threadIdx.x >> 5); row < n; row += warps) {
        const SRC* r = src + row * src_ld;
        float s = 0.f, e = 0.f;
        for (int c = lane; c < dp / 4; c += 32) {
            float4 v;
            const int c0 = c * 4;
            if (vec_ok && c0 + 3 < d) {
                v = load4_f32(r, c);
            } else {
                v.x = c0 + 0 < d ? to_f32(r[c0 + 0]) : 0.f;
                v.y = c0 + 1 < d ? to_f32(r[c0 + 1]) : 0.f;
                v.z = c0 + 2 < d ? to_f32(r[c0 + 2]) : 0.f;
                v.w = c0 + 3 < d ? to_f32(r[c0 + 3]) : 0.f;
            }
            float2 flo, fhi;
            uint2 packed;
            packed.x = pack_shadow2<FMT>(v.x, v.y, mbits, flo);
            packed.y = pack_shadow2<FMT>(v.z, v.w, mbits, fhi);
            if (shadow_is_master) v = make_float4(flo.x, flo.y, fhi.x, fhi.y);  // the rounded values ARE the row
            s = fmaf(v.x, v.x, s); s = fmaf(v.y, v.y, s); s = fmaf(v.z, v.z, s); s = fmaf(v.w, v.w, s);
            float dx = v.x - flo.x, dy = v.y - flo.y, dz = v.z - fhi.x, dw = v.w - fhi.y;
            e = fmaf(dx, dx, e); e = fmaf(dy, dy, e); e = fmaf(dz, dz, e); e = fmaf(dw, dw, e);
            if (dst_f32) reinterpret_cast<float4*>(dst_f32 + row * int64_t(dp))[c] = v;
            if (dst_h16) reinterpret_cast<uint2*>(dst_h16 + row * int64_t(dp))[c] = packed;
        }
        s = warp_sum(s);
        e = warp_sum(e);
        if (lane == 0) {
            if (norms2) norms2[row] = s;
            if (dnorms2) dnorms2[row] = e;
        }
        // NaN/Inf rows must not poison the bound: they can never be a valid neighbour anyway.
        if (s == s && s < FLT_MAX) wmax_n = fmaxf(wmax_n, s);
        if (e == e && e < FLT_MAX) wmax_d = fmaxf(wmax_d, e);
    }
    if (stats && lane == 0) {
        atomicMax(&stats->max_norm2, __float_as_uint(wmax_n));
        atomicMax(&stats->max_dnorm2, __float_as_uint(wmax_d));
    }
}

// eps[q]: bound on |approx score - exact score| for query q against ANY database row, where the
// approx score is the 16-bit x 16-bit -> fp32 tensor-core inner product (DESIGN.md "error bound"):
//   |<x^,y^> - <x,y>| <= |dx||y| + |x||dy| + |dx||dy|      (Cauchy-Schwarz, dx = x^ - x)
// plus a slack of dp * 2^-22 * |x||y| for the fp32 accumulation inside the MMA and the rerank.
// L2 compares keys 2<x,y> - |y|^2: the inner-product bound doubles, and fp32 roundings of order ulp(|y|^2) that no
// inner-product term sees are added, in units U = 2^-24 (|x|^2 + max|y|^2):
//   |y|^2 itself (ingest: a lane chains dp/32 FMAs, then 5 butterfly adds)            dp/32 + 5
//   the key fl(2 acc - |y|^2), |key| <= |x|^2 + 2|y|^2                                  2
//   the rescored distance fl(fl(|x|^2 + |y|^2) - 2a), |D| <= 2 (|x|^2 + |y|^2)          1 + 2
//   threshold = k-th key - 2 eps, lower = threshold + eps, lower - eps (values <= 2U)   3 x 2
// c(dp) = dp/32 + 16.  Negligible for normalised data (~6e-6 at dp = 1024 against eps ~1e-3); what it covers
// dominates when |x| << |y| or the data is 16-bit exact (eps = the slack alone), e.g. |y| / |x| = 4000 at dp = 64.
__global__ void query_eps_kernel(const float* __restrict__ xnorm2, const float* dnorm2, int64_t nq, int dp,
                                 const DbStats* __restrict__ stats, int metric, float* eps) {  // dnorm2 may alias eps
    int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const float ymax2 = __uint_as_float(stats->max_norm2);
    const float ymax = sqrtf(ymax2);
    const float dymax = sqrtf(__uint_as_float(stats->max_dnorm2));
    const float xn2 = xnorm2[q];
    const float xn = sqrtf(xn2);
    const float dx = sqrtf(dnorm2[q]);
    float e = dx * ymax + xn * dymax + dx * dymax + float(dp) * 2.384185791015625e-07f * xn * ymax;
    e *= 1.001f;
    if (metric == KNN_METRIC_L2) {
        e *= 2.f;  // approx score is 2<x,y> - |y|^2
        e += (float(dp) * 0.03125f + 16.f) * 5.9604644775390625e-08f * (xn2 + ymax2);
    }
    if (!(e == e) || e > FLT_MAX) e = FLT_MAX;
    eps[q] = e;
}

// ---------------------------------------------------------------------------------------
// Exact fp32 scan.  Per (row, query) pair: lane l accumulates elements 4c..4c+3 for
// c = l, l+32, ... in order with FMAs, then a butterfly sum - the rerank kernel repeats exactly
// this order, so a pair gets the same bits whichever path scored it.
template <int QT, int R, bool BF16DB>
__global__ void __launch_bounds__(kBlock)
scan_f32_kernel(const float* __restrict__ xq, const float* __restrict__ xnorm2, int64_t nq, int dp,
                const void* __restrict__ xb, const float* __restrict__ ynorm2, int64_t j0, int64_t j1, int metric,
                float* __restrict__ out, int64_t ld_out) {
    extern __shared__ float4 sq[];  // [QT][dp/4]
    const int dp4 = dp / 4;
    const int64_t q0 = int64_t(blockIdx.y) * QT;
    const int nqt = int((nq - q0) < QT ? (nq - q0) : QT);
    for (int i = threadIdx.x; i < QT * dp4; i += blockDim.x) {
        const int t = i / dp4, c = i - t * dp4;
        sq[i] = t < nqt ? reinterpret_cast<const float4*>(xq + (q0 + t) * int64_t(dp))[c]
                        : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warps = int64_t(gridDim.x) * kWarpsPerBlock;
    const int64_t wid = int64_t(blockIdx.x) * kWarpsPerBlock + (threadIdx.x >> 5);
    for (int64_t base = j0 + wid * R; base < j1; base += warps * R) {
        float acc[R][QT];
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int t = 0; t < QT; ++t) acc[r][t] = 0.f;
        for (int c = lane; c < dp4; c += 32) {
            float4 y[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int64_t row = base + r;
                if (row < j1) {
                    if (BF16DB) {
                        uint2 p = reinterpret_cast<const uint2*>(static_cast<const __nv_bfloat16*>(xb) +
                                                                 row * int64_t(dp))[c];
                        float2 a = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&p.x));
                        float2 b = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&p.y));
                        y[r] = make_float4(a.x, a.y, b.x, b.y);
                    } else {
                        y[r] = __ldg(reinterpret_cast<const float4*>(static_cast<const float*>(xb) +
                                                                     row * int64_t(dp)) + c);
                    }
                } else {
                    y[r] = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
#pragma unroll
            for (int t = 0; t < QT; ++t) {
                const float4 q = sq[t * dp4 + c];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    float a = acc[r][t];
                    a = fmaf(y[r].x, q.x, a); a = fmaf(y[r].y, q.y, a);
                    a = fmaf(y[r].z, q.z, a); a = fmaf(y[r].w, q.w, a);
                    acc[r][t] = a;
                }
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int64_t row = base + r;
            float mine = 0.f;
#pragma unroll
            for (int t = 0; t < QT; ++t) {
                const float v = warp_sum(acc[r][t]);
                if (lane == t) mine = v;
            }
            if (row < j1 && lane < nqt) {
                float v = mine;
                if (metric == KNN_METRIC_L2) {
                    v = xnorm2[q0 + lane] + ynorm2[row] - 2.0f * v;
                    v = v < 0.f ? 0.f : v;
                }
                out[(q0 + lane) * ld_out + (row - j0)] = v;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// A 4-element chunk of a database row as it lies in memory: the raw loads of a row are issued back to back and
// only converted when the FMAs consume them (a conversion next to its load makes every load wait for the previous one).
template <bool BF16DB> struct RowChunk { using T = float4; };
template <> struct RowChunk<true> { using T = uint2; };

__device__ __forceinline__ float4 chunk_to_f32(const float4& v) { return v; }
__device__ __forceinline__ float4 chunk_to_f32(const uint2& p) {
    // bf16 -> fp32 is a 16-bit shift
    return make_float4(__uint_as_float(p.x << 16), __uint_as_float(p.x & 0xFFFF0000u), __uint_as_float(p.y << 16),
                       __uint_as_float(p.y & 0xFFFF0000u));
}

// gridDim.y CTAs per query (1 for large batches; for small batches CTA y owns the list entries i with
// i % gridDim.y == y, so that a warp's serial chain of row fetches gets shorter and more SMs gather),
// the query row in shared memory.  Each warp takes 32 list entries at a time with one
// coalesced load, then walks the entries that passed the final threshold NR at a time (2 fp32 rows or 4 bf16
// rows: 8 KB in flight per warp either way): all loads of the NR rows are issued before the FMAs consume them.
// The FMA order per (row, query) pair is the scan kernel's, so a pair gets the same bits whichever path scored it.
//
// L2-blocked form (range_rows < number of rows): the grid is (row range, query) with the RANGE as the slow index, and
// a CTA rescoring only the candidates whose row lies in its range.  CTAs are dispatched in grid order, so at any time
// the resident CTAs of all SMs gather from one or two adjacent ranges of ~48 MB: a row crosses HBM once per query
// batch and is served from L2 to every other query that lists it.  With k = 1000 against 300k rows (C3) a batch lists
// every row ~59 times: 72 GB of row gathers per batch.
// MEASURED (profiles/r02_ncu_rerank_c3.md, r02_launches_c3_*_l2_blocked_rerank.md): it does what it says - DRAM reads
// 5.8 GB per batch instead of ~55 GB, L2 hit rate 88 % - and is 2 x SLOWER (18.9 vs 9.7 ms per batch): 409,600 CTAs of
// ~43 rows each run at 11.6 % warp occupancy, and the 80 GB that cross the L2->SM fabric per batch do so either way.
// HBM was never the limit of this kernel (the plain form already gathers at 7.4 TB/s, above the HBM roof, thanks to
// its L2 hits).  Off by default ("l2_blocked_rerank"); kept for databases whose rows are cold in HBM.
template <bool BF16DB, int NR, int U, int MINB>
__global__ void __launch_bounds__(kBlock, MINB)
rerank_kernel(const float* __restrict__ xq, const float* __restrict__ xnorm2, int dp, const void* __restrict__ xb,
              const float* __restrict__ ynorm2, int metric, float* __restrict__ cand_scores,
              uint32_t* __restrict__ cand_ids, const int* __restrict__ counts, const float* __restrict__ tau,
              int cap, unsigned nq, unsigned range_rows) {
    using Raw = typename RowChunk<BF16DB>::T;  // NR rows x U chunks per lane in flight
    extern __shared__ float4 sq[];  // [dp/4]
    const int64_t q = blockIdx.x % nq;
    const unsigned range = blockIdx.x / nq;
    const uint32_t id_lo = range * range_rows;                       // candidates of this CTA: id_lo <= id <= id_hi
    const uint32_t id_hi = range_rows >= kInvalidId - id_lo ? kInvalidId - 1u : id_lo + range_rows - 1u;
    const int dp4 = dp / 4;
    for (int i = threadIdx.x; i < dp4; i += blockDim.x)
        sq[i] = reinterpret_cast<const float4*>(xq + q * int64_t(dp))[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    int cnt = counts[q];
    cnt = cnt < cap ? cnt : cap;
    const float t = tau[q];
    float* cs = cand_scores + q * int64_t(cap);
    uint32_t* ci = cand_ids + q * int64_t(cap);
    const float xn = metric == KNN_METRIC_L2 ? xnorm2[q] : 0.f;
    const Raw* rows = static_cast<const Raw*>(xb);
    Raw zero;
    memset(&zero, 0, sizeof(zero));
    const bool mine = (lane % int(gridDim.y)) == int(blockIdx.y);  // no entry is touched by two CTAs
    for (int base = warp * 32; base < cnt; base += kWarpsPerBlock * 32) {
        const int i = base + lane;
        float approx = 0.f;
        uint32_t id = kInvalidId;
        bool here = false;  // this CTA decides the entry (it is touched by exactly one CTA: never rescored twice)
        if (i < cnt && mine) {
            id = ci[i];
            here = id >= id_lo && id <= id_hi;
            if (here) approx = cs[i];
        }
        const bool valid = here && (approx >= t);
        unsigned mask = __ballot_sync(0xffffffffu, valid);
        float res = 0.f;
        while (mask) {  // warp-uniform
            int src[NR];
            uint32_t rid[NR];
            const Raw* rp[NR];
            int n = 0;
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                src[r] = mask ? __ffs(int(mask)) - 1 : 0;
                n += mask ? 1 : 0;
                mask &= mask - 1;  // no-op when mask is already 0
                rid[r] = __shfl_sync(0xffffffffu, id, src[r]);
                rp[r] = rows + int64_t(rid[r]) * dp4;
            }
            float acc[NR];
#pragma unroll
            for (int r = 0; r < NR; ++r) acc[r] = 0.f;
            for (int c0 = lane; c0 < dp4; c0 += U * 32) {
                Raw y[NR][U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int c = c0 + u * 32;
#pragma unroll
                    for (int r = 0; r < NR; ++r) y[r][u] = (c < dp4 && r < n) ? __ldg(rp[r] + c) : zero;
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int c = c0 + u * 32;
                    if (c < dp4) {
                        const float4 qv = sq[c];
#pragma unroll
                        for (int r = 0; r < NR; ++r) {
                            const float4 yv = chunk_to_f32(y[r][u]);
                            float a = acc[r];
                            a = fmaf(yv.x, qv.x, a); a = fmaf(yv.y, qv.y, a);
                            a = fmaf(yv.z, qv.z, a); a = fmaf(yv.w, qv.w, a);
                            acc[r] = a;
                        }
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                float a = warp_sum(acc[r]);
                if (r < n) {
                    if (metric == KNN_METRIC_L2) {
                        a = xn + ynorm2[rid[r]] - 2.0f * a;
                        a = a < 0.f ? 0.f : a;
                    }
                    if (lane == src[r]) res = a;
                }
            }
        }
        if (here) {
            if (valid) cs[i] = res;
            else ci[i] = kInvalidId;
        }
    }
}

}  // namespace

int num_sms() {
    static int sms[64] = {};  // per device: the GPUs of one process need not be alike
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return 148;
    if (!sms[dev]) {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        sms[dev] = n > 0 ? n : 148;
    }
    return sms[dev];
}

// ---------------------------------------------------------------------------------------
int launch_normalize_l2(float* x, int64_t n, int64_t d, cudaStream_t s) {
    if (n <= 0 || d <= 0) return KNN_OK;
    const int vec_ok = (d % 4 == 0) && (reinterpret_cast<uintptr_t>(x) % 16 == 0);
    normalize_l2_kernel<<<grid_for_rows(n, kWarpsPerBlock, 8), kBlock, 0, s>>>(x, n, d, vec_ok);
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

// The vector loads need d % 4 == 0, a row stride that keeps every row aligned and an aligned base pointer: 16 bytes
// for fp32 rows, 8 bytes for 16-bit rows.  Anything else takes the scalar loads.
static int vec_loads_ok(const void* src, int64_t src_ld, int d, int src_dtype) {
    const uintptr_t align = src_dtype == KNN_DTYPE_F32 ? 16 : 8;
    return (d % 4 == 0) && (src_ld % 4 == 0) && (reinterpret_cast<uintptr_t>(src) % align == 0);
}

template <class SRC>
static void ingest_launch_t(int grid, const void* src, int64_t src_ld, int64_t n, int d, int dp, float* dst_f32,
                            h16_t* dst_h16, int fmt, float* norms2, float* dnorms2, DbStats* stats, int vec_ok,
                            int shadow_is_master, int mbits, cudaStream_t s) {
    const SRC* x = static_cast<const SRC*>(src);
    if (fmt == kFmtFP16)
        ingest_rows_kernel<kFmtFP16, SRC><<<grid, kBlock, 0, s>>>(x, src_ld, n, d, dp, dst_f32, dst_h16, norms2, dnorms2,
                                                                  stats, vec_ok, shadow_is_master, mbits);
    else
        ingest_rows_kernel<kFmtBF16, SRC><<<grid, kBlock, 0, s>>>(x, src_ld, n, d, dp, dst_f32, dst_h16, norms2, dnorms2,
                                                                  stats, vec_ok, shadow_is_master, mbits);
}

static int ingest_launch(const void* src, int src_dtype, int64_t src_ld, int64_t n, int d, int dp, float* dst_f32,
                         h16_t* dst_h16, int fmt, float* norms2, float* dnorms2, DbStats* stats, int shadow_is_master,
                         int mbits, cudaStream_t s) {
    const int vec_ok = vec_loads_ok(src, src_ld, d, src_dtype);
    const int grid = grid_for_rows(n, kWarpsPerBlock, 8);
    switch (src_dtype) {
        case KNN_DTYPE_F32:
            ingest_launch_t<float>(grid, src, src_ld, n, d, dp, dst_f32, dst_h16, fmt, norms2, dnorms2, stats, vec_ok,
                                   shadow_is_master, mbits, s);
            break;
        case KNN_DTYPE_F16:
            ingest_launch_t<__half>(grid, src, src_ld, n, d, dp, dst_f32, dst_h16, fmt, norms2, dnorms2, stats, vec_ok,
                                    shadow_is_master, mbits, s);
            break;
        case KNN_DTYPE_BF16:
            ingest_launch_t<__nv_bfloat16>(grid, src, src_ld, n, d, dp, dst_f32, dst_h16, fmt, norms2, dnorms2, stats,
                                           vec_ok, shadow_is_master, mbits, s);
            break;
        default:
            set_error("unknown source dtype %d", src_dtype);
            return KNN_ERR_INVALID;
    }
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

int launch_ingest(const void* src, int src_dtype, int64_t src_ld, int64_t n, int d, int dp, float* dst_f32, h16_t* dst_h16,
                  int fmt, int mbits, bool shadow_is_master, float* norms2, DbStats* stats, cudaStream_t s) {
    if (n <= 0) return KNN_OK;
    return ingest_launch(src, src_dtype, src_ld, n, d, dp, dst_f32, dst_h16, fmt, norms2, nullptr, stats,
                         shadow_is_master, mbits, s);
}

int launch_prep_queries(const void* xq, int xq_dtype, int64_t nq, int64_t nq_pad, int d, int dp, float* xq_f32,
                        h16_t* xq_h16, int fmt, int mbits, float* xnorm2, float* eps, const DbStats* stats, int metric,
                        cudaStream_t s) {
    if (nq <= 0) return KNN_OK;
    // eps doubles as scratch for |dx|^2 until query_eps_kernel overwrites it
    KNN_CHECK(ingest_launch(xq, xq_dtype, d, nq, d, dp, xq_f32, xq_h16, fmt, xnorm2, eps, nullptr, 0, mbits, s));
    if (xq_h16 && nq_pad > nq) {
        KNN_CHECK_CUDA(cudaMemsetAsync(xq_h16 + nq * int64_t(dp), 0, size_t(nq_pad - nq) * dp * sizeof(h16_t), s));
    }
    query_eps_kernel<<<int((nq + 255) / 256), 256, 0, s>>>(xnorm2, eps, nq, dp, stats, metric, eps);
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

template <int QT, bool BF16DB>
static int launch_scan_t(const float* xq_f32, const float* xnorm2, int64_t nq, int dp, const void* xb,
                         const float* ynorm2, int64_t j0, int64_t j1, int metric, float* out, int64_t ld_out,
                         cudaStream_t s) {
    constexpr int R = 4;
    auto kern = scan_f32_kernel<QT, R, BF16DB>;
    const size_t smem = size_t(QT) * dp * sizeof(float);
    KNN_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    const int64_t groups = (nq + QT - 1) / QT;
    // split so that (x blocks) * (query groups) covers the SMs a few times over
    int bx = grid_for_rows(j1 - j0, kWarpsPerBlock * R, 4);
    for (int64_t g0 = 0; g0 < groups; g0 += 32768) {
        const int64_t gn = groups - g0 < 32768 ? groups - g0 : 32768;
        dim3 grid(bx, unsigned(gn));
        kern<<<grid, kBlock, smem, s>>>(xq_f32 + g0 * QT * int64_t(dp), xnorm2 + g0 * QT, nq - g0 * QT, dp, xb,
                                        ynorm2, j0, j1, metric, out + g0 * QT * ld_out, ld_out);
        KNN_CHECK_LAUNCH();
    }
    return KNN_OK;
}

int launch_scan_f32(const float* xq_f32, const float* xnorm2, int64_t nq, int dp, const float* xb_f32,
                    const __nv_bfloat16* xb_bf16, const float* ynorm2, int64_t j0, int64_t j1, int metric,
                    float* out, int64_t ld_out, cudaStream_t s) {
    if (nq <= 0 || j1 <= j0) return KNN_OK;
    // QT queries stay in shared memory (QT * dp * 4 bytes): 8 for dp <= 6144, fewer beyond.
    const bool bf = xb_f32 == nullptr;
    const void* xb = bf ? static_cast<const void*>(xb_bf16) : static_cast<const void*>(xb_f32);
    const size_t per_q = size_t(dp) * sizeof(float);
    int qt = 8;
    while (qt > 1 && per_q * qt > 200 * 1024) qt >>= 1;
    if (per_q * qt > 200 * 1024) {
        set_error("dimension %d too large for the scan kernel", dp);
        return KNN_ERR_LIMIT;
    }
#define KNN_SCAN_CASE(QT)                                                                                   \
    case QT:                                                                                                \
        return bf ? launch_scan_t<QT, true>(xq_f32, xnorm2, nq, dp, xb, ynorm2, j0, j1, metric, out, ld_out, s) \
                  : launch_scan_t<QT, false>(xq_f32, xnorm2, nq, dp, xb, ynorm2, j0, j1, metric, out, ld_out, s);
    switch (qt) {
        KNN_SCAN_CASE(8)
        KNN_SCAN_CASE(4)
        KNN_SCAN_CASE(2)
        KNN_SCAN_CASE(1)
    }
#undef KNN_SCAN_CASE
    return KNN_ERR_INVALID;
}

int launch_rerank(const float* xq_f32, const float* xnorm2, int64_t nq, int dp, const float* xb_f32,
                  const __nv_bfloat16* xb_bf16, const float* ynorm2, int metric, float* cand_scores,
                  uint32_t* cand_ids, const int* counts, const float* tau, int cap, int64_t ntotal, int k, int l2_blocked,
                  cudaStream_t s) {
    if (nq <= 0) return KNN_OK;
    const size_t smem = size_t(dp) * sizeof(float);
    // fewer queries than a couple of CTAs per SM: every list is shared by `split` CTAs (a power of two <= 8)
    int split = 1;
    while (split < 8 && nq * split < 2 * int64_t(num_sms())) split *= 2;
    // L2-blocked (see the kernel): when the batch lists every row several times (nq k > 4 N) and the rows do not fit
    // L2 anyway, walk the database in ranges of ~48 MB of rows
    const int64_t row_bytes = int64_t(dp) * (xb_f32 ? 4 : 2);
    int64_t range_rows = int64_t(1) << 32;
    int64_t n_ranges = 1;
    if (l2_blocked && split == 1 && nq * int64_t(k) > 4 * ntotal && ntotal * row_bytes > (int64_t(64) << 20)) {
        range_rows = std::max<int64_t>(1024, (int64_t(48) << 20) / row_bytes);
        n_ranges = (ntotal + range_rows - 1) / range_rows;
        if (n_ranges * nq > 0x7FFFFFFFll) {
            range_rows = int64_t(1) << 32;
            n_ranges = 1;
        }
    }
    const dim3 grid = dim3(unsigned(nq * n_ranges), unsigned(split), 1);
    const unsigned rr = range_rows >= (int64_t(1) << 32) ? 0xFFFFFFFFu : unsigned(range_rows);
#define KNN_RERANK(BF, NRV, UV, MINBV, XB)                                                                             \
    {                                                                                                                  \
        auto kern = rerank_kernel<BF, NRV, UV, MINBV>;                                                                 \
        KNN_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));            \
        kern<<<grid, kBlock, smem, s>>>(xq_f32, xnorm2, dp, XB, ynorm2, metric, cand_scores, cand_ids, counts, tau, cap, unsigned(nq), rr); \
    }
    // 8 KB in flight per warp either way.  Measured on B200 (4M x 1024 fp32 rows, 16384 queries, k = 1000): 2 x 8, 4 x 4,
    // 4 x 8 and 2 x 4 (rows x chunks) with 1-4 CTAs per SM all take 23.1-24.2 ms - the gather of 4 KB rows is not
    // limited by bytes in flight or occupancy.
    if (xb_f32) {
        KNN_RERANK(false, 2, 8, 1, xb_f32)
    } else {
        KNN_RERANK(true, 4, 8, 1, xb_bf16)
    }
#undef KNN_RERANK
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

}  // namespace knn

// Distance GEMM with a fused threshold-filter epilogue for sm_100a: TMA (128-byte swizzle) ->
// shared memory -> tcgen05.mma (16-bit x 16-bit -> fp32 in TMEM; bf16 or fp16 per operand) -> tcgen05.ld -> compare against
// the per-query candidate threshold -> rare append to the per-query candidate list.  The
// nq x N score matrix never reaches HBM.
//
// This is the one dense contraction of the flat-search path: the `sgemm` inside faiss's
// knn_inner_product / knn_L2sqr behind index.search (reference call sites cath/search.py:24,
// pfam/proteins_search.py:49, seqvec_search/main.py:45; faiss itself is third-party, see
// oracle/flat_oracle.py).  Scores produced here are approximate (16-bit inputs); the candidate
// threshold carries the error bound and the survivors are rescored in fp32 (rerank_kernel).
//
// Tile per CTA: 128 queries (TMEM lanes) x 256 database rows (TMEM columns) x 64 (one 128-byte
// swizzle atom of K per pipeline stage).  Two variants of the same kernel:
//   CG = 1  one CTA per tile, tcgen05.mma.cta_group::1, M = 128, 4 stages of 48 KB;
//   CG = 2  a CTA pair (cluster of 2) per 256 x 256 tile, tcgen05.mma.cta_group::2, M = 256: each
//           CTA stages its 128 query rows and HALF of the database tile (128 rows), the pair's
//           tensor cores read both halves -> half the database bytes per CTA, 6 stages of 32 KB.
// Warp roles: 0..3 = epilogue (one TMEM lane quarter each), 4 = TMA producer, 5 = MMA issuer
// (+ TMEM allocator; leader CTA only issues).  Persistent CTAs, static tile schedule with the
// query tile fastest so that co-resident CTAs share database tiles in L2.
#include <cuda.h>

#include <type_traits>

#include "common.cuh"

namespace knn {

namespace {

constexpr int BM = 128;   // query rows per CTA
constexpr int BN = 256;   // database rows per tile
constexpr int BK = 64;
constexpr int kMaxStages = 6;
constexpr int kAccStages = 2;
constexpr int kTmemCols = 512;
constexpr int kThreads = 192;
// Warp roles.  The SM sub-partition arbiter favours the higher warp id among eligible warps, and warp w lives
// on sub-partition w % 4: the two single-thread issuers (TMA, MMA) sit ABOVE the epilogue warps they share a
// scheduler with, otherwise an ALU-busy epilogue warp starves the MMA issuer and the tensor pipe drains.
constexpr int kProducerWarp = 4;
constexpr int kMmaWarp = 5;
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;  // clears the CTA-rank bit of a shared::cluster address -> even CTA of the pair

template <int CG>
struct Cfg {
    // measured on B200: for the CTA pair 4, 5 and 6 stages of 32 KB run the same
    static constexpr int kStages = 4;
    static constexpr int kRowsB = BN / CG;  // database rows staged by one CTA
    static constexpr uint32_t kBytesA = BM * BK * 2;
    static constexpr uint32_t kBytesB = kRowsB * BK * 2;
    static constexpr uint32_t kBytesStage = kBytesA + kBytesB;
    static constexpr size_t smem_bytes(int stages) {
        return size_t(stages) * kBytesStage + 1024 /*align slack*/ + 256 /*barriers*/ + 4 * (512 * 8 + 8 * 32 * 16) + 16 /*EpilogueSmem*/;
    }
    static constexpr size_t kSmemBytes = smem_bytes(kStages);
    // kind::f16 instruction descriptor: D = F32 (bits 4-5 = 1), A format at bits 7-9 and B format at bits 10-12
    // (0 = F16, 1 = BF16, chosen per launch: the operands' 16-bit formats are independent of each other),
    // both K-major (bits 15, 16 = 0), N >> 3 at bits 17-22, M >> 4 at bits 24-28 (M = 256 for a CTA pair).
    static constexpr uint32_t kInstrDescBase = (1u << 4) | (uint32_t(BN >> 3) << 17) | (uint32_t((BM * CG) >> 4) << 24);
    static uint32_t instr_desc(int fmt_a, int fmt_b) {
        return kInstrDescBase | ((fmt_a == kFmtBF16 ? 1u : 0u) << 7) | ((fmt_b == kFmtBF16 ? 1u : 0u) << 10);
    }
};

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// L2 eviction-priority policies (the encodings CUTLASS passes as TMA cache hints)
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;  // database tiles: streamed once per query batch
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;   // query tiles: re-read for every database tile
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(
            smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(hint)
        : "memory");
}
// CTA-pair variant: both CTAs load into their own shared memory, the bytes are accounted on the
// LEADER CTA's barrier (peer bit cleared), where the MMA issuer waits.
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(
            smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "l"(hint)
        : "memory");
}
// Multicast form: the box lands at the same shared-memory offset in every CTA of `mask`, and each destination's bytes
// are accounted on the barrier (same offset, peer bit cleared) of the LEADER of that destination's CTA pair.
__device__ __forceinline__ void tma_load_2d_pair_mc(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, uint16_t mask,
                                                    uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster.L2::cache_hint"
        " [%0], [%1, {%4, %5}], [%2], %3, %6;" ::"r"(smem_u32(smem_dst)),
        "l"(map), "r"(smem_u32(bar) & kPeerBitMask), "h"(mask), "r"(c0), "r"(c1), "l"(hint)
        : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
    uint32_t raddr;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(smem_u32(bar)), "r"(cta));
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(raddr) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t cols) {
    if constexpr (CG == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    if constexpr (CG == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
    } else {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
    }
}

// D[tmem] (+)= A[smem] * B[smem]^T: one (128*CG) x 256 x 16 MMA of 16-bit operands (CG = 2: across the CTA pair)
template <int CG>
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    if constexpr (CG == 1) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
            "}\n" ::"r"(tmem_d),
            "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
            "}\n" ::"r"(tmem_d),
            "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
            : "memory");
    }
}
// arrives on the mbarrier (CG = 2: on the barrier at this offset in BOTH CTAs of the pair) once all
// MMAs issued so far by this thread have completed
template <int CG>
__device__ __forceinline__ void umma_commit(uint64_t* bar, uint16_t mask = 3) {
    if constexpr (CG == 1) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
    } else {  // arrives on the barrier at this offset in every CTA of `mask` (default: the two CTAs of a lone pair)
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                         smem_u32(bar)),
                     "h"(mask)
                     : "memory");
    }
}

__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand tile in shared memory, 128-byte swizzle: rows are 128 B apart, 8-row groups
// (one swizzle atom, 1024 B) are contiguous -> stride byte offset 1024; the leading byte offset
// is unused for swizzled K-major layouts.  Bits: [0,14) addr>>4, [16,30) LBO>>4, [32,46) SBO>>4,
// [46,48) version = 1 (sm_100), [61,64) layout = 2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= uint64_t((saddr & 0x3FFFF) >> 4);
    d |= uint64_t(1) << 16;
    d |= uint64_t(1024 >> 4) << 32;
    d |= uint64_t(1) << 46;
    d |= uint64_t(2) << 61;
    return d;
}

struct __align__(8) Barriers {
    uint64_t full[kMaxStages];
    uint64_t empty[kMaxStages];
    uint64_t acc_full[kAccStages];
    uint64_t acc_empty[kAccStages];
    uint32_t tmem_base;
};

struct GemmArgs {
    int64_t nq;        // real queries (rows >= nq of the padded query matrix are ignored)
    int m_tiles;       // nq_pad / (128 * CG)
    int n_tiles;       // ceil((j1 - j0) / 256)
    int num_kb;        // dp / 64
    int64_t j0, j1;    // database rows of this panel
    const float* ynorm2;
    float* thr;
    int* counts;
    float* cand_scores;
    uint32_t* cand_ids;
    int cap;
    uint64_t hint_q, hint_db;  // L2 eviction-priority policies of the two TMA streams
    int stages;                // shared-memory pipeline depth
    uint32_t idesc;            // tcgen05 instruction descriptor (operand formats of this launch)
    int debug_skip_epilogue;   // experiments only: accumulators are not read (results are then meaningless)
};
// Arguments of the filtered instantiations: the unfiltered ones keep GemmArgs (and their code) as it is.
struct GemmArgsFilt : GemmArgs {
    RowFilter filt;            // rows that may not become candidates (exclude: one id per query of the launch)
};
template <bool FILT> using GemmArgsT = typename std::conditional<FILT, GemmArgsFilt, GemmArgs>::type;

// Eligibility bits of the 32 columns j_first .. j_first + 31 for a query that excludes row ex_row (-1: none).
__device__ __forceinline__ uint32_t eligible_cols(const RowFilter& f, int64_t j_first, int64_t ex_row) {
    uint32_t m = allow_word(f, j_first);
    const int64_t e = ex_row - j_first;
    if (e >= 0 && e < 32) m &= ~(1u << int(e));
    return m;
}
__device__ __forceinline__ float nan_score() { return __uint_as_float(0x7FC00000u); }

constexpr int kStashEntries = 512;  // per epilogue warp: (score bits, lane << 8 | column in tile)

struct EpilogueSmem {                 // one slice per epilogue warp
    uint2 stash[4][kStashEntries];    // survivors waiting to be appended to the global candidate lists
    float4 dump[4][8 * 32];           // the 32 scores of every lane of a flagged column group ([j/4][lane])
    int count[4];                     // entries in the stash (may run past kStashEntries: overflow went direct)
};

// Appends the stashed survivors of one warp to the per-query candidate lists.  Four entries per lane
// are in flight so that the atomics' round trips overlap.
__device__ __forceinline__ void drain_stash(const uint2* stash, int n, int lane, int64_t q_warp0, int64_t jbase,
                                            const GemmArgs& args) {
    for (int e0 = 0; e0 < n; e0 += 128) {
        uint2 ent[4];
        int pos[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int e = e0 + u * 32 + lane;
            pos[u] = -1;
            if (e < n) {
                ent[u] = stash[e];
                pos[u] = atomicAdd(args.counts + (q_warp0 + (ent[u].y >> 8)), 1);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (pos[u] >= 0 && pos[u] < args.cap) {
                const int64_t q = q_warp0 + (ent[u].y >> 8);
                args.cand_scores[q * int64_t(args.cap) + pos[u]] = __uint_as_float(ent[u].x);
                args.cand_ids[q * int64_t(args.cap) + pos[u]] = uint32_t(jbase + (ent[u].y & 255u));
            }
        }
    }
}

__device__ __forceinline__ void append_direct(uint2 ent, int64_t q_warp0, int64_t jbase, const GemmArgs& args) {
    const int64_t q = q_warp0 + (ent.y >> 8);
    const int pos = atomicAdd(args.counts + q, 1);
    if (pos < args.cap) {
        args.cand_scores[q * int64_t(args.cap) + pos] = __uint_as_float(ent.x);
        args.cand_ids[q * int64_t(args.cap) + pos] = uint32_t(jbase + (ent.y & 255u));
    }
}

template <bool L2>
__device__ __forceinline__ void load_scores(uint32_t taddr, int64_t j_first, const GemmArgs& args, float (&v)[32]) {
    uint32_t r[32];
    tmem_ld_32x32b_x32(taddr, r);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        v[i] = __uint_as_float(r[i]);
        if (L2) {
            const int64_t j = j_first + i;
            v[i] = 2.0f * v[i] - (j < args.j1 ? __ldg(args.ynorm2 + j) : 0.f);
        }
    }
}

template <int CG, bool L2, bool DENSE, bool FILT>
__global__ void __launch_bounds__(kThreads, 1)
gemm_filter_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_db, const GemmArgsT<FILT> args) {
    using C = Cfg<CG>;
    const int nstages = args.stages;  // depth of the TMA -> MMA shared-memory ring (<= kMaxStages)
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment for the 128B-swizzle atoms; plain pointer arithmetic keeps the shared address space
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    Barriers* bars = reinterpret_cast<Barriers*>(smem + size_t(nstages) * C::kBytesStage);
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_tiles = args.m_tiles * args.n_tiles;
    const uint32_t cta_rank = CG == 1 ? 0u : cluster_ctarank();  // position in the CTA pair
    const bool leader = cta_rank == 0;
    const int unit = CG == 1 ? blockIdx.x : (blockIdx.x >> 1);   // tile-scheduling unit (CTA or CTA pair)
    const int num_units = CG == 1 ? gridDim.x : (gridDim.x >> 1);

    if (warp == kProducerWarp && lane == 0) {
        prefetch_tmap(&map_q);
        prefetch_tmap(&map_db);
        for (int i = 0; i < nstages; ++i) {
            mbar_init(&bars->full[i], 1);
            mbar_init(&bars->empty[i], 1);
        }
        for (int i = 0; i < kAccStages; ++i) {
            mbar_init(&bars->acc_full[i], 1);
            mbar_init(&bars->acc_empty[i], 4 * CG);  // one arrival per epilogue warp of every CTA on the tile
        }
        fence_barrier_init();
    }
    if (warp == kMmaWarp) tmem_alloc<CG>(&bars->tmem_base, kTmemCols);
    tc_fence_before();
    if constexpr (CG == 1) __syncthreads(); else cluster_sync_all();  // peer barriers must exist before anyone signals them
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;

    if (warp == kProducerWarp) {
        // ===== TMA producer (every CTA loads its own query rows and its share of the database tile) =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = unit; tile < num_tiles; tile += num_units) {
                const int mt = tile % args.m_tiles;
                const int nt = tile / args.m_tiles;
                const int row_q = mt * (BM * CG) + int(cta_rank) * BM;
                const int row_db = int(args.j0) + nt * BN + int(cta_rank) * C::kRowsB;
                for (int kb = 0; kb < args.num_kb; ++kb) {
                    mbar_wait(&bars->empty[stage], phase ^ 1);
                    uint8_t* sa = smem + size_t(stage) * C::kBytesStage;
                    uint8_t* sb = sa + C::kBytesA;
                    if constexpr (CG == 1) {
                        mbar_expect_tx(&bars->full[stage], C::kBytesStage);
                        tma_load_2d(sa, &map_q, &bars->full[stage], kb * BK, row_q, args.hint_q);
                        tma_load_2d(sb, &map_db, &bars->full[stage], kb * BK, row_db, args.hint_db);
                    } else {
                        if (leader) mbar_expect_tx(&bars->full[stage], C::kBytesStage * 2);  // both CTAs' bytes
                        tma_load_2d_pair(sa, &map_q, &bars->full[stage], kb * BK, row_q, args.hint_q);
                        tma_load_2d_pair(sb, &map_db, &bars->full[stage], kb * BK, row_db, args.hint_db);
                    }
                    if (++stage == nstages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        // ===== MMA issuer (one thread; for a CTA pair only the leader issues, for both CTAs) =====
        if (lane == 0 && leader) {
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int tile = unit; tile < num_tiles; tile += num_units) {
                mbar_wait(&bars->acc_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + uint32_t(acc * BN);
                for (int kb = 0; kb < args.num_kb; ++kb) {
                    mbar_wait(&bars->full[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + size_t(stage) * C::kBytesStage);
                    const uint32_t sb = sa + C::kBytesA;
                    const uint64_t da = make_smem_desc(sa);
                    const uint64_t db = make_smem_desc(sb);
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) {
                        // advance 16 elements (32 B) along K inside the swizzle atom: +2 in 16-byte units
                        umma_f16<CG>(tmem_d, da + uint64_t(k * 2), db + uint64_t(k * 2), args.idesc, (kb | k) ? 1u : 0u);
                    }
                    umma_commit<CG>(&bars->empty[stage]);  // smem slot reusable once these MMAs have read it
                    if (++stage == nstages) { stage = 0; phase ^= 1; }
                }
                umma_commit<CG>(&bars->acc_full[acc]);  // accumulator complete -> epilogue (of both CTAs)
                if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===== epilogue: warps 0..3, TMEM lane quarter = warp =====
        const int quarter = warp & 3;
        int acc = 0;
        uint32_t acc_phase = 0;
        EpilogueSmem* es = reinterpret_cast<EpilogueSmem*>(smem + size_t(nstages) * C::kBytesStage + 256);
        uint2* stash = es->stash[warp];
        float4* dump = es->dump[warp];
        int* stash_count = &es->count[warp];
        if (lane == 0) *stash_count = 0;
        __syncwarp();
        for (int tile = unit; tile < num_tiles; tile += num_units) {
            const int mt = tile % args.m_tiles;
            const int nt = tile / args.m_tiles;
            const int64_t q = int64_t(mt) * (BM * CG) + int64_t(cta_rank) * BM + quarter * 32 + lane;
            const int64_t jbase = args.j0 + int64_t(nt) * BN;
            const bool q_ok = q < args.nq;
            const float thr = q_ok ? args.thr[q] : FLT_MAX;
            int64_t ex_row = -1;  // lane-local
            if constexpr (FILT) ex_row = q_ok ? excluded_row(args.filt, q) : -1;
            mbar_wait(&bars->acc_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + uint32_t(acc * BN) + (uint32_t(quarter * 32) << 16);
            const int64_t q_warp0 = q - lane;  // query of lane 0 of this warp
#ifdef KNN_EXPERIMENTS
            // measurement aids (never compiled into the shipped library): 1 main loop only, 2 TMEM reads only,
            // 3 TMEM reads + threshold compares with the survivors ignored
            if (args.debug_skip_epilogue == 1) {
            } else if (args.debug_skip_epilogue == 2) {
                uint32_t sink = 0;
#pragma unroll 1
                for (int cg = 0; cg < BN / 32; ++cg) {
                    uint32_t r[32];
                    tmem_ld_32x32b_x32(taddr + uint32_t(cg * 32), r);
                    tmem_ld_wait();
                    sink ^= r[0] ^ r[31];
                }
                if (sink == 0x7fc12345u) args.counts[0] = 1;
            } else if (args.debug_skip_epilogue == 3) {
                uint32_t flagged = 0;
#pragma unroll 1
                for (int cg = 0; cg < BN / 32; ++cg) {
                    float v[32];
                    load_scores<L2>(taddr + uint32_t(cg * 32), jbase + cg * 32, args, v);
                    bool any = false;
#pragma unroll
                    for (int i = 0; i < 32; ++i) any |= (v[i] >= thr);
                    if (__any_sync(0xffffffffu, any)) flagged |= 1u << cg;
                }
                if (flagged == 0xdeadbeefu) args.counts[0] = 1;
            } else
#endif
            if constexpr (DENSE) {
#pragma unroll 1
                for (int cg = 0; cg < BN / 32; ++cg) {
                    float v[32];
                    load_scores<L2>(taddr + uint32_t(cg * 32), jbase + cg * 32, args, v);
                    const int64_t j_first = jbase + cg * 32;
                    // ineligible columns: a NaN score and an invalid id, which tighten and rerank skip and never count
                    uint32_t ok = ~0u;
                    if constexpr (FILT) {
                        ok = eligible_cols(args.filt, j_first, ex_row);
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] = ((ok >> i) & 1u) ? v[i] : nan_score();
                    }
                    auto col_id = [&](int i) { return FILT && !((ok >> i) & 1u) ? kInvalidId : uint32_t(j_first + i); };
                    if (q_ok) {
                        float* cs = args.cand_scores + q * int64_t(args.cap) + (j_first - args.j0);
                        uint32_t* ci = args.cand_ids + q * int64_t(args.cap) + (j_first - args.j0);
                        if (j_first + 32 <= args.j1) {
#pragma unroll
                            for (int i = 0; i < 32; i += 4) {
                                *reinterpret_cast<float4*>(cs + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
                                *reinterpret_cast<uint4*>(ci + i) = make_uint4(col_id(i), col_id(i + 1), col_id(i + 2), col_id(i + 3));
                            }
                        } else {
#pragma unroll
                            for (int i = 0; i < 32; ++i) {
                                if (j_first + i < args.j1) {
                                    cs[i] = v[i];
                                    ci[i] = col_id(i);
                                }
                            }
                        }
                    }
                    __syncwarp();  // reconverge before the next warp-wide tcgen05.ld
                }
            } else {
                // One compare per score (LDTM + 16 FMNMX3 + FSETP + vote per 32 columns).  A column group in
                // which some lane has a survivor (rare once the threshold has tightened) takes the side path:
                // the lanes' scores are dumped to shared memory, each lane builds its 32-bit survivor mask and
                // walks its set bits, parking (score, lane, column) in the warp's stash.  The stash is appended
                // to the global candidate lists only after the TMEM stage has been handed back to the MMA
                // issuer, so atomics and stores run under the next tile's MMAs.
#pragma unroll 1
                for (int cg = 0; cg < BN / 32; ++cg) {
                    float v[32];
                    load_scores<L2>(taddr + uint32_t(cg * 32), jbase + cg * 32, args, v);
                    bool any = false;
#pragma unroll
                    for (int i = 0; i < 32; ++i) any |= (v[i] >= thr);
                    if (__any_sync(0xffffffffu, any)) {  // warp-uniform
#pragma unroll
                        for (int t = 0; t < 8; ++t)
                            dump[t * 32 + lane] = make_float4(v[4 * t], v[4 * t + 1], v[4 * t + 2], v[4 * t + 3]);
                        uint32_t mask = 0;
                        if (any) {
#pragma unroll
                            for (int i = 0; i < 32; ++i) mask |= (v[i] >= thr) ? (1u << i) : 0u;
                            const int64_t left = args.j1 - (jbase + cg * 32);  // columns of this group inside the panel
                            if (left < 32) mask &= left <= 0 ? 0u : ((1u << int(left)) - 1u);
                            // the group's bitmap word is the same for the whole warp; the exclusion is this lane's
                            if constexpr (FILT) mask &= eligible_cols(args.filt, jbase + cg * 32, ex_row);
                        }
                        while (mask) {  // a lane reads back only what it dumped itself
                            const int i = __ffs(int(mask)) - 1;
                            mask &= mask - 1;
                            const float val = reinterpret_cast<const float*>(dump + (i >> 2) * 32 + lane)[i & 3];
                            const uint2 ent = make_uint2(__float_as_uint(val), (uint32_t(lane) << 8) | uint32_t(cg * 32 + i));
                            const int slot = atomicAdd(stash_count, 1);
                            if (slot < kStashEntries) stash[slot] = ent;
                            else append_direct(ent, q_warp0, jbase, args);  // stash full (dense early panels)
                        }
                        __syncwarp();
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                // the accumulator stage may be overwritten once every epilogue warp of every CTA on this
                // tile has drained it; the MMA issuer waits on the leader's barrier
                if constexpr (CG == 1) mbar_arrive(&bars->acc_empty[acc]);
                else mbar_arrive_remote(&bars->acc_empty[acc], 0);
            }
            {
                __syncwarp();
                int nst = *stash_count;  // same value in every lane
                if (nst) {
                    nst = nst < kStashEntries ? nst : kStashEntries;
                    drain_stash(stash, nst, lane, q_warp0, jbase, args);
                    __syncwarp();
                    if (lane == 0) *stash_count = 0;
                }
            }
            if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
        }
    }

    tc_fence_before();
    // nobody may leave (or free TMEM) while the peer can still read this CTA's shared memory or signal its barriers
    if constexpr (CG == 1) __syncthreads(); else cluster_sync_all();
    if (warp == kMmaWarp) {
        tc_fence_after();
        tmem_dealloc<CG>(tmem_base, kTmemCols);
    }
}

// =============================================================================================
// Few-queries variant (<= 64 queries per launch): the roles of the operands are swapped.  The database rows are the
// M = 128 operand and stream through a deep TMA ring, 16 KB per stage, ALL of it database bytes; the queries are the
// N operand (NQT = 32 or 64 rows) and stay resident in shared memory for the whole launch.  With one query tile the
// main kernel re-loads the query tile into every stage (half of its bytes in flight) and spends a 256 x 256 MMA on
// a handful of queries; here a launch is a pure stream of the 16-bit rows: the bandwidth kernel of the path.
// Accumulator: 128 TMEM lanes = database rows, NQT columns = queries; an epilogue thread owns one database row and
// compares its NQT scores with the per-query thresholds (shared memory).
constexpr int SBM = 128;            // database rows per CTA and tile
constexpr int kStreamAcc = 4;       // accumulator stages of NQT columns
constexpr int kStreamMaxStages = 10;
constexpr uint32_t kStreamBytesA = SBM * BK * 2;

struct StreamBarriers {
    uint64_t full[kStreamMaxStages];
    uint64_t empty[kStreamMaxStages];
    uint64_t acc_full[kStreamAcc];
    uint64_t acc_empty[kStreamAcc];
    uint64_t queries;
    uint32_t tmem_base;
};

// nq_cta: query rows resident per CTA (NQT for one CTA, NQT / 2 for a CTA pair)
// (filt: plus the excluded row of each of the up to 128 queries)
static size_t stream_smem_bytes(int nq_cta, int num_kb, int stages, bool filt) {
    return 1024 /*align slack*/ + size_t(num_kb) * nq_cta * BK * 2 + size_t(stages) * kStreamBytesA + sizeof(StreamBarriers) + 128 * sizeof(float) + 64 +
           (filt ? 128 * sizeof(int64_t) : 0);
}

// CG = 2 (NQT = 128): a CTA pair works on 256 database rows with tcgen05.mma.cta_group::2 (M = 256, N = 128).  Each
// CTA streams ITS 128 rows and keeps HALF of the queries resident (64 rows = 128 KB at d = 1024, what one CTA holds
// for NQT = 64): the pair's tensor cores read both halves of the N operand, so 128 queries cost no more shared memory
// per SM than 64 - and the launch stays a pure stream of database bytes where the main kernel would pad the batch to
// a 256-query tile pair and re-load the query tile with every stage.
//
// NP = 2 (NQT = 128 per pair, 256 queries in all): a cluster of FOUR CTAs = two such pairs on the SAME 256 database
// rows, pair p scoring queries [128 p, 128 p + 128).  The database half-tile a CTA needs is the one its counterpart
// in the other pair needs (ranks {0, 2} rows 0..127, ranks {1, 3} rows 128..255), so each of the two loads half of it
// (64 rows) and TMA-multicasts it to both: the rows cross HBM and L2 once for 256 queries, every SM still does the MMA
// work of a 128-query launch, and no query tile is ever re-loaded - where the main kernel, for 129..256 queries, keeps
// the tensor pipe 98 % busy, re-loads its query tile with every stage and runs into the power cap (DESIGN.md 5c).
// A stage slot may be refilled once BOTH pairs have consumed it (the refill writes into both), hence empty barriers
// that count one commit per pair, multicast to all four CTAs.
// MEASURED (256 queries x 10M rows, whole call): correct (bit-identical, tests/test_gpu_parity.py), but 7.4 ms against
// the main kernel's 6.0 ms - and the arithmetic says why no form of it can reach the HBM roof: a cluster RECEIVES
// 64 KB per K block for 32 KB of unique rows, so streaming unique rows at HBM speed needs every SM to take a 16 KB
// stage per 0.19 us, exactly the time its MMAs for that stage take at the full clock.  256 queries are the machine
// balance; under the power cap (1.3-1.4 GHz) the tensor pipe sets the pace, and the multicast loads' longer latency on a
// 6-stage ring costs the rest.  Off by default ("stream_quad"); kept because it is the measured answer to "would
// multicast help".
template <int NQT, bool L2, bool DENSE, int CG, int NP, bool FILT>
__global__ void __launch_bounds__(kThreads, 1)
gemm_stream_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_db, const GemmArgsT<FILT> args) {
    static_assert(NP == 1 || CG == 2, "two pairs need CTA pairs");
    constexpr int NQ_CTA = NQT / CG;                 // query rows staged by one CTA
    constexpr uint32_t kTmemColsS = NQT * kStreamAcc < 32 ? 32 : NQT * kStreamAcc;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int nstages = args.stages;
    const uint32_t bytes_q_kb = NQ_CTA * BK * 2;                    // one K block of this CTA's resident queries
    uint8_t* smem_q = smem;                                         // [num_kb][NQ_CTA x 64] 128-byte swizzled
    uint8_t* smem_a = smem + size_t(args.num_kb) * bytes_q_kb;      // [nstages][128 x 64]
    StreamBarriers* bars = reinterpret_cast<StreamBarriers*>(smem_a + size_t(nstages) * kStreamBytesA);
    float* thr_s = reinterpret_cast<float*>(bars + 1);
    int64_t* ex_s = reinterpret_cast<int64_t*>(thr_s + 128);  // FILT: row each query excludes (-1: none)
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_tiles = args.n_tiles;  // tiles of 128 * CG database rows
    const uint32_t cl_rank = CG == 1 ? 0u : cluster_ctarank();       // rank in the cluster (0..CG * NP - 1)
    const uint32_t pair = cl_rank >> 1;                               // which CTA pair of the cluster
    const uint32_t cta_rank = cl_rank & 1u;                           // position inside the pair
    const bool leader = cta_rank == 0;
    const int unit = blockIdx.x / (CG * NP);                          // tile-scheduling unit = cluster
    const int num_units = gridDim.x / (CG * NP);
    const int q_base = int(pair) * NQT;                               // first query of this pair
    const uint16_t pair_mask = uint16_t(3u << (2 * pair));           // the two CTAs of this pair
    const uint16_t all_mask = uint16_t((1u << (CG * NP)) - 1u);     // every CTA of the cluster
    // instruction descriptor: M = 128 * CG, N = NQT
    const uint32_t idesc = (args.idesc & ~((0x3Fu << 17) | (0x1Fu << 24))) | (uint32_t(NQT >> 3) << 17) | (uint32_t((SBM * CG) >> 4) << 24);

    if (warp == kProducerWarp && lane == 0) {
        prefetch_tmap(&map_q);
        prefetch_tmap(&map_db);
        for (int i = 0; i < nstages; ++i) {
            mbar_init(&bars->full[i], 1);
            mbar_init(&bars->empty[i], NP);  // one commit per pair that reads (a copy of) the slot
        }
        for (int i = 0; i < kStreamAcc; ++i) {
            mbar_init(&bars->acc_full[i], 1);
            mbar_init(&bars->acc_empty[i], 4 * CG);
        }
        mbar_init(&bars->queries, 1);
        fence_barrier_init();
    }
    if (warp == kMmaWarp) tmem_alloc<CG>(&bars->tmem_base, kTmemColsS);
    if (threadIdx.x < 128)
        thr_s[threadIdx.x] = (threadIdx.x < NQT && q_base + int(threadIdx.x) < args.nq) ? args.thr[q_base + threadIdx.x] : FLT_MAX;
    if constexpr (FILT) {
        if (threadIdx.x < 128)
            ex_s[threadIdx.x] = (threadIdx.x < NQT && q_base + int(threadIdx.x) < args.nq) ? excluded_row(args.filt, q_base + threadIdx.x) : -1;
    }
    tc_fence_before();
    if constexpr (CG == 1) __syncthreads(); else cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;

    if (warp == kProducerWarp) {
        if (lane == 0) {
            // resident queries: this CTA's share of the N operand
            if constexpr (CG == 1) {
                mbar_expect_tx(&bars->queries, uint32_t(args.num_kb) * bytes_q_kb);
                for (int kb = 0; kb < args.num_kb; ++kb)
                    tma_load_2d(smem_q + size_t(kb) * bytes_q_kb, &map_q, &bars->queries, kb * BK, 0, args.hint_q);
            } else {
                if (leader) mbar_expect_tx(&bars->queries, uint32_t(args.num_kb) * bytes_q_kb * 2);
                for (int kb = 0; kb < args.num_kb; ++kb)
                    tma_load_2d_pair(smem_q + size_t(kb) * bytes_q_kb, &map_q, &bars->queries, kb * BK, q_base + int(cta_rank) * NQ_CTA,
                                     args.hint_q);
            }
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = unit; tile < num_tiles; tile += num_units) {
                const int row_db = int(args.j0) + tile * (SBM * CG) + int(cta_rank) * SBM;
                for (int kb = 0; kb < args.num_kb; ++kb) {
                    mbar_wait(&bars->empty[stage], phase ^ 1);
                    if constexpr (CG == 1) {
                        mbar_expect_tx(&bars->full[stage], kStreamBytesA);
                        tma_load_2d(smem_a + size_t(stage) * kStreamBytesA, &map_db, &bars->full[stage], kb * BK, row_db, args.hint_db);
                    } else if constexpr (NP == 1) {
                        if (leader) mbar_expect_tx(&bars->full[stage], kStreamBytesA * 2);
                        tma_load_2d_pair(smem_a + size_t(stage) * kStreamBytesA, &map_db, &bars->full[stage], kb * BK, row_db, args.hint_db);
                    } else {
                        // this CTA's half (64 rows) of the 128 rows it shares with rank ^ 2, multicast to both; every leader
                        // expects the 2 x 16 KB that land in its own pair
                        if (leader) mbar_expect_tx(&bars->full[stage], kStreamBytesA * 2);
                        tma_load_2d_pair_mc(smem_a + size_t(stage) * kStreamBytesA + size_t(pair) * (kStreamBytesA / 2), &map_db,
                                            &bars->full[stage], kb * BK, row_db + int(pair) * (SBM / 2),
                                            uint16_t(0x5u << cta_rank), args.hint_db);
                    }
                    if (++stage == nstages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        if (lane == 0 && leader) {
            mbar_wait(&bars->queries, 0);
            tc_fence_after();
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int tile = unit; tile < num_tiles; tile += num_units) {
                mbar_wait(&bars->acc_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + uint32_t(acc * NQT);
                for (int kb = 0; kb < args.num_kb; ++kb) {
                    mbar_wait(&bars->full[stage], phase);
                    tc_fence_after();
                    const uint64_t da = make_smem_desc(smem_u32(smem_a + size_t(stage) * kStreamBytesA));
                    const uint64_t db = make_smem_desc(smem_u32(smem_q + size_t(kb) * bytes_q_kb));
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k)
                        umma_f16<CG>(tmem_d, da + uint64_t(k * 2), db + uint64_t(k * 2), idesc, (kb | k) ? 1u : 0u);
                    umma_commit<CG>(&bars->empty[stage], NP == 1 ? pair_mask : all_mask);
                    if (++stage == nstages) { stage = 0; phase ^= 1; }
                }
                umma_commit<CG>(&bars->acc_full[acc], pair_mask);
                if (++acc == kStreamAcc) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===== epilogue: warp w owns database rows 32 w .. 32 w + 31 of this CTA's half of the tile (TMEM lanes) =====
        int acc = 0;
        uint32_t acc_phase = 0;
        const int nq = int(args.nq - q_base < NQT ? (args.nq - q_base < 0 ? 0 : args.nq - q_base) : NQT);  // real queries of this pair
        for (int tile = unit; tile < num_tiles; tile += num_units) {
            const int64_t j = args.j0 + int64_t(tile) * (SBM * CG) + int64_t(cta_rank) * SBM + warp * 32 + lane;  // this thread's database row
            const bool row_ok = j < args.j1;
            bool row_in = true;  // the selector's bit of this lane's row
            if constexpr (FILT) row_in = row_ok && row_allowed(args.filt, j);
            float yn = 0.f;
            if (L2 && row_ok) yn = __ldg(args.ynorm2 + j);
            mbar_wait(&bars->acc_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + uint32_t(acc * NQT) + (uint32_t(warp * 32) << 16);
#pragma unroll 1
            for (int c0 = 0; c0 < NQT; c0 += 32) {
                uint32_t r[32];
                tmem_ld_32x32b_x32(taddr + uint32_t(c0), r);
                tmem_ld_wait();
                if (c0 < nq && row_ok) {
                    if (DENSE) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) {
                            if (c0 + i < nq) {  // lanes of a warp hold consecutive rows: coalesced per query
                                float v = __uint_as_float(r[i]);
                                if (L2) v = 2.0f * v - yn;
                                uint32_t id = uint32_t(j);
                                if (FILT && !(row_in && ex_s[c0 + i] != j)) {  // ineligible: skipped by tighten and rerank
                                    v = nan_score();
                                    id = kInvalidId;
                                }
                                args.cand_scores[int64_t(q_base + c0 + i) * args.cap + (j - args.j0)] = v;
                                args.cand_ids[int64_t(q_base + c0 + i) * args.cap + (j - args.j0)] = id;
                            }
                        }
                    } else {
                        uint32_t mask = 0;
#pragma unroll
                        for (int i = 0; i < 32; ++i) {
                            float v = __uint_as_float(r[i]);
                            if (L2) v = 2.0f * v - yn;
                            r[i] = __float_as_uint(v);
                            mask |= (v >= thr_s[c0 + i] && (!FILT || ex_s[c0 + i] != j)) ? (1u << i) : 0u;  // padding queries carry +FLT_MAX
                        }
                        if (!row_in) mask = 0u;
                        while (mask) {  // rare once the thresholds have tightened
                            const int i = __ffs(int(mask)) - 1;
                            mask &= mask - 1;
                            float v = 0.f;
#pragma unroll
                            for (int u = 0; u < 32; ++u) v = (u == i) ? __uint_as_float(r[u]) : v;  // no dynamic register indexing
                            const int64_t q = q_base + c0 + i;
                            const int pos = atomicAdd(args.counts + q, 1);
                            if (pos < args.cap) {
                                args.cand_scores[q * int64_t(args.cap) + pos] = v;
                                args.cand_ids[q * int64_t(args.cap) + pos] = uint32_t(j);
                            }
                        }
                    }
                }
                __syncwarp();  // reconverge before the next warp-wide tcgen05.ld
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (CG == 1) mbar_arrive(&bars->acc_empty[acc]);
                else mbar_arrive_remote(&bars->acc_empty[acc], pair * 2);  // the leader of this pair
            }
            if (++acc == kStreamAcc) { acc = 0; acc_phase ^= 1; }
        }
    }

    tc_fence_before();
    if constexpr (CG == 1) __syncthreads(); else cluster_sync_all();
    if (warp == kMmaWarp) {
        tc_fence_after();
        tmem_dealloc<CG>(tmem_base, kTmemColsS);
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

struct GemmPlan {
    EncodeTiledFn encode = nullptr;
    int sms = 148;
    int cta_group = 2;  // 1: one CTA per tile, 2: CTA pairs (tcgen05 cta_group::2)
    int l2_hints = 0;   // 1: queries evict-last, database evict-first
    int debug_skip_epilogue = 0;
    int stages = 0;     // 0: default depth (4)
    int stream_kernel = 1;  // launches with <= 64 queries use the few-queries variant (database rows as the M operand)
    int stream_pair = 1;    // launches with 65..128 queries use the CTA-pair form of the few-queries variant
    int stream_quad = 0;    // experiments: 129..256 queries on its two-pair (cluster of 4, multicast) form - measured slower
    int small_m128 = 0;     // experiments: launches with 65..128 queries use the single-CTA (M = 128) variant of the main kernel
};

void gemm_plan_set_cta_group(GemmPlan* p, int cg) { p->cta_group = cg == 1 ? 1 : 2; }
void gemm_plan_set_l2_hints(GemmPlan* p, int on) { p->l2_hints = on; }
void gemm_plan_set_debug(GemmPlan* p, int skip_epilogue) { p->debug_skip_epilogue = skip_epilogue; }
void gemm_plan_set_stages(GemmPlan* p, int stages) { p->stages = stages; }
void gemm_plan_set_stream_kernel(GemmPlan* p, int on) { p->stream_kernel = on; }
void gemm_plan_set_small_m128(GemmPlan* p, int on) { p->small_m128 = on; }
void gemm_plan_set_stream_pair(GemmPlan* p, int on) { p->stream_pair = on; }
void gemm_plan_set_stream_quad(GemmPlan* p, int on) { p->stream_quad = on; }
int gemm_plan_query_rows_multiple(const GemmPlan* p) { return BM * p->cta_group; }

int gemm_plan_create(GemmPlan** out, int device) {
    GemmPlan* p = new GemmPlan();
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
        cudaGetLastError();
        set_error("cuTensorMapEncodeTiled is not available from the driver");
        delete p;
        return KNN_ERR_CUDA;
    }
    p->encode = reinterpret_cast<EncodeTiledFn>(fn);
    int major = 0;
    cudaDeviceGetAttribute(&p->sms, cudaDevAttrMultiProcessorCount, device);
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
    if (major != 10) {
        set_error("the tensor-core path needs an sm_100 device (found compute capability %d.x)", major);
        delete p;
        return KNN_ERR_CUDA;
    }
    *out = p;
    return KNN_OK;
}

void gemm_plan_destroy(GemmPlan* p) { delete p; }

// The tensor map only moves 16-bit elements (zero fill out of bounds): one map type serves bf16 and fp16 rows.
static int make_map(GemmPlan* p, CUtensorMap* map, const h16_t* base, int64_t rows, int dp, int box_rows) {
    cuuint64_t gdim[2] = {cuuint64_t(dp), cuuint64_t(rows)};
    cuuint64_t gstride[1] = {cuuint64_t(dp) * 2};
    cuuint32_t box[2] = {cuuint32_t(BK), cuuint32_t(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = p->encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<h16_t*>(base), gdim, gstride, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld, dp=%d)", int(r), (long long)rows, dp);
        return KNN_ERR_CUDA;
    }
    return KNN_OK;
}

template <int CG, bool L2, bool DENSE, bool FILT>
static int launch_variant(GemmPlan* p, const CUtensorMap& map_q, const CUtensorMap& map_db, const GemmArgsFilt& af, cudaStream_t s) {
    const GemmArgsT<FILT> a = af;
    auto kern = gemm_filter_kernel<CG, L2, DENSE, FILT>;
    static bool attr_done[64] = {};  // per instantiation and device (function attributes are per device)
    int dev = 0;
    KNN_CHECK_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_done[dev]) {
        KNN_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            int(Cfg<CG>::smem_bytes(CG == 1 ? 4 : kMaxStages))));
        // The SM's shared-memory carveout is picked from a few sizes when the (persistent) CTA lands and cannot change
        // while it is resident: with the default the 162 KB of the 4-stage ring select the 164 KB configuration and
        // nothing else that uses shared memory fits next to it (tools/micro/overlap_test.cu).  Asking for the largest
        // carveout leaves ~64 KB for the rescoring / selection kernels of the previous query batch, which run on a
        // side stream under this kernel (index.cu: search_tensor).
        KNN_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        if (dev >= 0 && dev < 64) attr_done[dev] = true;
    }
    const int64_t tiles = int64_t(a.m_tiles) * a.n_tiles;
    const int units_max = p->sms / CG;
    const int units = int(tiles < units_max ? tiles : units_max);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(unsigned(units * CG), 1, 1);
    cfg.blockDim = dim3(kThreads, 1, 1);
    cfg.dynamicSmemBytes = Cfg<CG>::smem_bytes(a.stages);
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    KNN_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, map_q, map_db, a));
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

template <int NQT, bool L2, bool DENSE, int CG, int NP, bool FILT>
static int launch_stream_variant(GemmPlan* p, const CUtensorMap& map_q, const CUtensorMap& map_db, const GemmArgsFilt& af, size_t smem,
                                 cudaStream_t s) {
    const GemmArgsT<FILT> a = af;
    auto kern = gemm_stream_kernel<NQT, L2, DENSE, CG, NP, FILT>;
    static bool attr_done[64] = {};
    int dev = 0;
    KNN_CHECK_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_done[dev]) {
        KNN_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        if (dev >= 0 && dev < 64) attr_done[dev] = true;
    }
    int units_max = p->sms / (CG * NP);
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(kThreads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG * NP;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (NP > 1) {  // clusters of 4 must fit inside a GPC: ask how many can be resident at once (persistent grid)
        static int max_clusters[64] = {};
        if (dev >= 0 && dev < 64 && !max_clusters[dev]) {
            cfg.gridDim = dim3(unsigned(units_max * CG * NP), 1, 1);
            int n = 0;
            KNN_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
            max_clusters[dev] = n > 0 ? n : 1;
        }
        if (dev >= 0 && dev < 64 && max_clusters[dev] < units_max) units_max = max_clusters[dev];
    }
    const int units = a.n_tiles < units_max ? a.n_tiles : units_max;
    cfg.gridDim = dim3(unsigned(units * CG * NP), 1, 1);
    KNN_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, map_q, map_db, a));
    KNN_CHECK_LAUNCH();
    return KNN_OK;
}

// Few-queries launch: returns KNN_OK and sets *done when the stream kernel took the launch.
static int try_stream_launch(GemmPlan* p, const h16_t* xq_h16, int fmt, int64_t nq, int64_t nq_pad, int dp, const h16_t* xb_h16,
                             int64_t ntotal, const float* ynorm2, int64_t j0, int64_t j1, int metric, bool dense_first,
                             FilterState st, const RowFilter& filt, cudaStream_t s, bool* done) {
    *done = false;
    if (!p->stream_kernel || nq > 256 || nq_pad < 256 || dp % BK != 0) return KNN_OK;
    if (nq > 64 && !p->stream_pair) return KNN_OK;
    if (nq > 128 && !p->stream_quad) return KNN_OK;
    const int np = nq > 128 ? 2 : 1;    // 129..256 queries: two CTA pairs per cluster, 128 queries each
    const int nqt = nq <= 32 ? 32 : (nq <= 64 ? 64 : 128);
    const int cg = nqt == 128 ? 2 : 1;  // 128 queries: a CTA pair, each CTA keeps 64 of them resident
    const int nq_cta = nqt / cg;
    const int num_kb = dp / BK;
    const bool filtered = filt.active();
    int stages = kStreamMaxStages;
    while (stages >= 4 && stream_smem_bytes(nq_cta, num_kb, stages, filtered) > size_t(227 * 1024)) --stages;
    if (stages < 4) return KNN_OK;  // the resident queries leave no room for a ring: the main kernel takes it
    CUtensorMap map_q, map_db;
    KNN_CHECK(make_map(p, &map_q, xq_h16, nq_pad, dp, nq_cta));
    KNN_CHECK(make_map(p, &map_db, xb_h16, ntotal, dp, np == 2 ? SBM / 2 : SBM));  // two pairs: each CTA loads half of its rows
    GemmArgsFilt a;
    a.nq = nq;
    a.m_tiles = 1;
    a.n_tiles = int((j1 - j0 + SBM * cg - 1) / (SBM * cg));
    a.num_kb = num_kb;
    a.j0 = j0;
    a.j1 = j1;
    a.ynorm2 = ynorm2;
    a.thr = st.thr;
    a.counts = st.counts;
    a.cand_scores = st.cand_scores;
    a.cand_ids = st.cand_ids;
    a.cap = st.cap;
    a.debug_skip_epilogue = 0;
    a.idesc = Cfg<1>::instr_desc(fmt, fmt);
    a.stages = stages;
    a.hint_q = kEvictNormal;
    a.hint_db = kEvictNormal;
    a.filt = filt;
    const size_t smem = stream_smem_bytes(nq_cta, num_kb, stages, filtered);
    const bool l2 = metric == KNN_METRIC_L2;
    *done = true;
#define KNN_STREAM_DISPATCH(NQTV, CGV, NPV, F)                                                                         \
    if (l2) {                                                                                                          \
        return dense_first ? launch_stream_variant<NQTV, true, true, CGV, NPV, F>(p, map_q, map_db, a, smem, s)        \
                           : launch_stream_variant<NQTV, true, false, CGV, NPV, F>(p, map_q, map_db, a, smem, s);      \
    } else {                                                                                                           \
        return dense_first ? launch_stream_variant<NQTV, false, true, CGV, NPV, F>(p, map_q, map_db, a, smem, s)       \
                           : launch_stream_variant<NQTV, false, false, CGV, NPV, F>(p, map_q, map_db, a, smem, s);     \
    }
    if (filtered) {
        if (np == 2) { KNN_STREAM_DISPATCH(128, 2, 2, true) }
        if (nqt == 32) { KNN_STREAM_DISPATCH(32, 1, 1, true) } else if (nqt == 64) { KNN_STREAM_DISPATCH(64, 1, 1, true) } else { KNN_STREAM_DISPATCH(128, 2, 1, true) }
    }
    if (np == 2) { KNN_STREAM_DISPATCH(128, 2, 2, false) }
    if (nqt == 32) { KNN_STREAM_DISPATCH(32, 1, 1, false) } else if (nqt == 64) { KNN_STREAM_DISPATCH(64, 1, 1, false) } else { KNN_STREAM_DISPATCH(128, 2, 1, false) }
#undef KNN_STREAM_DISPATCH
}

int gemm_filter_launch(GemmPlan* p, const h16_t* xq_h16, int fmt_q, int64_t nq, int64_t nq_pad, int dp,
                       const h16_t* xb_h16, int fmt_db, int64_t ntotal, const float* ynorm2, int64_t j0, int64_t j1,
                       int metric, bool dense_first, FilterState st, const RowFilter& filt, cudaStream_t s) {
    if (j1 <= j0 || nq <= 0) return KNN_OK;
    // small_m128 (experiments, off): 65..128 queries on single-CTA tiles (M = 128) instead of padding them to a CTA
    // pair's M = 256.  Measured slower (4 stages of 48 KB cover less latency than the pair's 6 x 32 KB).
    const int cg = (p->cta_group == 2 && nq <= BM && p->small_m128) ? 1 : p->cta_group;
    if (dp % BK != 0 || nq_pad % (BM * cg) != 0) {
        set_error("gemm_filter: dp (%d) must be a multiple of %d and nq_pad (%lld) of %d", dp, BK, (long long)nq_pad, BM * cg);
        return KNN_ERR_INVALID;
    }
    if (dense_first && j1 - j0 > st.cap) {
        set_error("gemm_filter: dense panel larger than the candidate capacity");
        return KNN_ERR_INVALID;
    }
    if (fmt_q == fmt_db) {
        bool done = false;
        KNN_CHECK(try_stream_launch(p, xq_h16, fmt_q, nq, nq_pad, dp, xb_h16, ntotal, ynorm2, j0, j1, metric, dense_first, st, filt, s, &done));
        if (done) return KNN_OK;
    }
    CUtensorMap map_q, map_db;
    KNN_CHECK(make_map(p, &map_q, xq_h16, nq_pad, dp, BM));
    KNN_CHECK(make_map(p, &map_db, xb_h16, ntotal, dp, BN / cg));
    GemmArgsFilt a;
    a.nq = nq;
    a.m_tiles = int(nq_pad / (BM * cg));
    a.n_tiles = int((j1 - j0 + BN - 1) / BN);
    a.num_kb = dp / BK;
    a.j0 = j0;
    a.j1 = j1;
    a.ynorm2 = ynorm2;
    a.thr = st.thr;
    a.counts = st.counts;
    a.cand_scores = st.cand_scores;
    a.cand_ids = st.cand_ids;
    a.cap = st.cap;
    a.debug_skip_epilogue = p->debug_skip_epilogue;
    a.idesc = cg == 1 ? Cfg<1>::instr_desc(fmt_q, fmt_db) : Cfg<2>::instr_desc(fmt_q, fmt_db);
    a.stages = cg == 1 ? Cfg<1>::kStages : Cfg<2>::kStages;
    // Few query tiles: the kernel is the bandwidth kernel of small batches (the database streams by once) and what
    // limits it is bytes in flight - half of every stage is the re-loaded query tile.  6 stages instead of 4:
    // 5.3 -> 5.8 TB/s at nq = 1, 4.5 -> 4.8 TB/s at nq = 256 (profiles/r01_small_batch.md); equal for large batches.
    if (cg == 2 && a.m_tiles <= 4) a.stages = kMaxStages;
    if (p->stages >= 2 && p->stages <= (cg == 1 ? 4 : kMaxStages)) a.stages = p->stages;
    a.hint_q = p->l2_hints ? kEvictLast : kEvictNormal;
    a.hint_db = p->l2_hints ? kEvictFirst : kEvictNormal;
    a.filt = filt;
    const bool l2 = metric == KNN_METRIC_L2;
#define KNN_GEMM_DISPATCH(CGV, F)                                                                     \
    if (l2) {                                                                                         \
        return dense_first ? launch_variant<CGV, true, true, F>(p, map_q, map_db, a, s)               \
                           : launch_variant<CGV, true, false, F>(p, map_q, map_db, a, s);             \
    } else {                                                                                          \
        return dense_first ? launch_variant<CGV, false, true, F>(p, map_q, map_db, a, s)              \
                           : launch_variant<CGV, false, false, F>(p, map_q, map_db, a, s);            \
    }
    if (filt.active()) {
        if (cg == 1) { KNN_GEMM_DISPATCH(1, true) } else { KNN_GEMM_DISPATCH(2, true) }
    }
    if (cg == 1) { KNN_GEMM_DISPATCH(1, false) } else { KNN_GEMM_DISPATCH(2, false) }
#undef KNN_GEMM_DISPATCH
}

}  // namespace knn

// mma_common.cuh -- what the tcgen05 search kernels share: tile constants, PTX wrappers
// (mbarrier, TMA, tcgen05.mma / .ld / .commit, TMEM allocation), UMMA descriptors, raw candidate
// lists and the host-side TMA descriptor builder.  Included by search_mma.cu and search_mma_small.cu.
#pragma once

#include "index.cuh"

#include <cuda.h>
#include <algorithm>
#include <cstdlib>

namespace ivr {

constexpr int kMmaThreads   = 384;                 // 4 control warps + 2 epilogue sets of 4 warps
constexpr int kTileN        = 256;                 // DB rows per tile (UMMA N)
constexpr int kTileQ        = 128;                 // queries per CTA (UMMA M per CTA)
constexpr int kKBlock       = 64;                  // fp16 per 128-byte swizzle row
constexpr int kQBlockBytes  = kTileQ * 128;        // one k-block of the query tile: 16 KB
constexpr int kMaxKBlocks   = 8;                   // dpad <= 512 keeps the query tile resident
constexpr int kSmemBudget   = 227 * 1024;
constexpr int kBarrierBytes = 1024;

// ---------------------------------------------------------------- PTX wrappers ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_local(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive on the barrier at the same offset in CTA `cta` of the cluster.  Relaxed: the only thing
// the waiter (the MMA issuer) consumes is TMEM, ordered by tcgen05.wait::ld + tcgen05.fence.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t cta) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(bar), "r"(cta) : "memory");
}
// try_wait with a suspend-time hint (same value CUTLASS uses): the thread is put to sleep by the
// hardware until the phase completes instead of polling -- the producer / MMA-issuer / epilogue
// warps share warp schedulers, and a polling waiter steals issue slots (and power) from the
// warps that have work.
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity), "r"(0x989680u) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) { }
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after()  { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int CG>
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int x, int y,
                                            uint64_t policy) {
    if constexpr (CG == 1) {
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
            " [%0], [%1, {%3, %4}], [%2], %5;"
            ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(x), "r"(y), "l"(policy) : "memory");
    } else {
        // both CTAs of the pair signal the LEADER's barrier (peer bit cleared)
        asm volatile(
            "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
            " [%0], [%1, {%3, %4}], [%2], %5;"
            ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar & 0xFEFFFFFFu), "r"(x), "r"(y), "l"(policy)
            : "memory");
    }
}
// L2 eviction-priority descriptors (same encodings as cute::TMA::CacheHintSm90)
constexpr uint64_t kL2EvictNormal = 0x1000000000000000ull;
constexpr uint64_t kL2EvictFirst  = 0x12F0000000000000ull;
constexpr uint64_t kL2EvictLast   = 0x14F0000000000000ull;
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

template <int CG>
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    if constexpr (CG == 1) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
    }
}
// arrive on `bar` (in every CTA of the group) once all previously issued MMAs have completed
template <int CG>
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    if constexpr (CG == 1) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
    } else {
        asm volatile(
            "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
            ::"r"(bar), "h"(static_cast<uint16_t>(3)) : "memory");
    }
}
template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
    if constexpr (CG == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    if constexpr (CG == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
    else
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
// wait for every outstanding tcgen05.ld; the registers are in/out operands so that no use of
// them can be scheduled above the wait
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&v)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
        : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
          "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
          "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
          "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
        :: "memory");
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
//   [0,14) start address >> 4, [16,30) leading byte offset >> 4 (unused for swizzled K-major: 1),
//   [32,46) stride byte offset >> 4 (8 rows x 128 B = 1024 B), [46,48) version = 1 (Blackwell),
//   [61,64) layout type = 2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    return static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) |
           (static_cast<uint64_t>(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor (cute::UMMA::InstrDescriptor): D = F32 (bits 4-5 = 1),
// A = B = F16 (bits 7-9, 10-12 = 0), both K-major (bits 15, 16 = 0), N >> 3 at [17,23), M >> 4 at [24,29).
__host__ __device__ constexpr uint32_t make_idesc(int m, int n) {
    return (1u << 4) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

// ------------------------------------------------------------------- the kernel ----
// Candidate lists of this kernel hold RAW pairs {score bits (lo), row (hi)} so that an append is
// one predicated 8-byte store; compaction converts to ordered keys and back.
__device__ __forceinline__ uint64_t raw_to_key(uint64_t raw) {
    return make_key(__uint_as_float(static_cast<uint32_t>(raw)), static_cast<uint32_t>(raw >> 32));
}
__device__ __forceinline__ uint64_t key_to_raw(uint64_t key) {
    return static_cast<uint64_t>(__float_as_uint(key_score(key))) | (static_cast<uint64_t>(key_row(key)) << 32);
}

// Warp-cooperative EXACT compaction of a RAW list to its k best (sorted descending, still raw);
// returns the k-th best score (or -inf when the list holds fewer than k entries).  Entry i of the
// list lives at list[i * stride] (stride 1: contiguous; 32: one of a warp's interleaved lists).
template <int E>
__device__ __forceinline__ float warp_compact_raw(uint64_t* list, int cnt, int k, int cap, int lane, int stride = 1) {
    if constexpr (E > 0) {
        uint64_t v[E];
#pragma unroll
        for (int j = 0; j < E; ++j) {
            const int g = j * 32 + lane;
            v[j] = (g < cnt) ? raw_to_key(list[static_cast<int64_t>(g) * stride]) : 0ull;
        }
        warp_sort_desc<E>(v, lane);
        __syncwarp();
        uint64_t kth = 0;
#pragma unroll
        for (int j = 0; j < E; ++j) {
            const int g = lane * E + j;
            if (g < k && g < cnt) list[static_cast<int64_t>(g) * stride] = key_to_raw(v[j]);
            if (g == k - 1) kth = v[j];
        }
        kth = __shfl_sync(0xffffffffu, kth, (k - 1) / E);
        __syncwarp();
        return (cnt >= k) ? key_score(kth) : __int_as_float(0xff800000);
    } else {
        for (int g = lane; g < cnt; g += 32) list[static_cast<int64_t>(g) * stride] = raw_to_key(list[static_cast<int64_t>(g) * stride]);
        __syncwarp();
        const float t = warp_compact_topk_mem(list, cnt, k, cap, lane, stride);
        const int keep = min(cnt, k);
        for (int g = lane; g < keep; g += 32) list[static_cast<int64_t>(g) * stride] = key_to_raw(list[static_cast<int64_t>(g) * stride]);
        __syncwarp();
        return t;
    }
}

// ---- lane-parallel pruning of a warp's 32 INTERLEAVED candidate lists ------------------------
// In the batched kernels every epilogue THREAD owns one query's list; entry i of lane l lives at
// warp_block[i * 32 + l], so the 32 lanes walk their lists in lockstep with coalesced accesses.
// A list does not need its exact k best to make room -- any pivot score with at least k entries
// strictly above it is a valid admission threshold (the final k-th best is above it), and
// everything at or below the pivot can be dropped.  Each lane sorts 16 samples of its list in
// registers, counts its entries against 8 candidate pivots around the expected rank of the k-th
// best in ONE pass, adopts the highest pivot that still has k entries above it and filters the
// list in place.  All 32 lists are pruned in the time the warp-cooperative sort needs for a
// fraction of one (measured: ~10 us per list for the sort; the 32 lists of a warp used to be
// compacted one after the other, which was the whole cold-start cost of a search).
constexpr int kListStride = 32;

__device__ __forceinline__ void sort16_desc(float (&s)[16]) {
#pragma unroll
    for (int sz = 2; sz <= 16; sz <<= 1) {
#pragma unroll
        for (int t = sz >> 1; t >= 1; t >>= 1) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int p = j ^ t;
                if (p > j) {
                    const bool desc = (j & sz) == 0;
                    const float a = s[j], b = s[p];
                    const float mx = fmaxf(a, b), mn = fminf(a, b);
                    s[j] = desc ? mx : mn;
                    s[p] = desc ? mn : mx;
                }
            }
        }
    }
}

__device__ __forceinline__ float raw_score(uint64_t raw) { return __uint_as_float(static_cast<uint32_t>(raw)); }

// my_list: entry 0 of this lane's list.  Lanes holding fewer than k + 16 entries sit the round out.
// On return cnt / tau are updated; the result is the mask of lanes that wanted pruning but found no
// pivot (heavy ties) -- the caller compacts those exactly.
__device__ __forceinline__ unsigned warp_prune_lists(uint64_t* my_list, int& cnt, float& tau, int k) {
    const float NEG_INF = __int_as_float(0xff800000);
    const bool act = cnt >= k + 16;
    const int cmax = __reduce_max_sync(0xffffffffu, act ? cnt : 0);
    if (cmax == 0) return 0u;
    float s[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {                              // samples spread evenly over the list
        const int i = act ? ((2 * j + 1) * cnt) >> 5 : 0;
        s[j] = act ? raw_score(my_list[static_cast<int64_t>(i) * kListStride]) : NEG_INF;
    }
    sort16_desc(s);
    const float s_min = s[15];
    // candidate pivots: the samples of rank sh .. sh + 7, sh + 2 ~ the rank with k entries above it
    const int j0 = act ? (16 * k + cnt - 1) / cnt : 0;
    const int sh = max(0, min(j0 - 2, 8));
#pragma unroll
    for (int b = 0; b < 4; ++b) {                               // per-lane shift by sh (register barrel shifter)
        const bool on = (sh >> b) & 1;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const int src = (j + (1 << b) < 16) ? j + (1 << b) : 15;
            s[j] = on ? s[src] : s[j];
        }
    }
    int c[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) c[j] = 0;
    for (int i0 = 0; i0 < cmax; i0 += 8) {                       // 8 independent loads in flight per round
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
            v[u] = (act && i0 + u < cnt) ? raw_score(my_list[static_cast<int64_t>(i0 + u) * kListStride]) : NEG_INF;
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
            for (int j = 0; j < 8; ++j) c[j] += (v[u] > s[j]) ? 1 : 0;
    }
    float pv = NEG_INF; bool ok = false;
#pragma unroll
    for (int j = 7; j >= 0; --j)
        if (c[j] >= k) { pv = s[j]; ok = true; }                // ends on the HIGHEST pivot with >= k entries above it
    unsigned retry = __ballot_sync(0xffffffffu, act && !ok);
    if (retry) {                                                // unlucky sample: fall back to the lowest sample
        int c2 = 0;
        const bool mine = act && !ok;
        const int cmax2 = __reduce_max_sync(0xffffffffu, mine ? cnt : 0);
        for (int i = 0; i < cmax2; ++i)
            c2 += (mine && i < cnt && raw_score(my_list[static_cast<int64_t>(i) * kListStride]) > s_min) ? 1 : 0;
        if (mine && c2 >= k) { pv = s_min; ok = true; }
    }
    const bool doit = act && ok;
    const int cmax3 = __reduce_max_sync(0xffffffffu, doit ? cnt : 0);
    int w = 0;
    for (int i0 = 0; i0 < cmax3; i0 += 8) {                      // in-place filter; 8 loads in flight, then the stores
        uint64_t e[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
            e[u] = (doit && i0 + u < cnt) ? my_list[static_cast<int64_t>(i0 + u) * kListStride] : 0ull;
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if (doit && i0 + u < cnt && raw_score(e[u]) > pv) { my_list[static_cast<int64_t>(w) * kListStride] = e[u]; ++w; }
    }
    if (doit) { cnt = w; tau = fmaxf(tau, pv); }
    return __ballot_sync(0xffffffffu, act && !ok);
}

// ------------------------------------------------------------------ host side ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// 2-D fp16 row-major [rows, cols] tensor, box = [box_rows, 64 cols], 128-byte swizzle
static int make_tmap(CUtensorMap* map, const void* base, int64_t rows, int cols, int box_rows) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return IVR_ECUDA; }
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(cols) * 2};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(kKBlock), static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", static_cast<int>(r)); return IVR_ECUDA; }
    return IVR_OK;
}

static int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return (e && *e) ? atoi(e) : dflt;
}

// ---- shared by the batched, the small-batch and the range host paths (defined in search_mma.cu) ----
int launch_queries_to_f16(const float* q, __half* out, float* scale, uint32_t* tau_g, int64_t nq, int64_t nq_pad,
                          int dim, int dpad, cudaStream_t st);
// The TMA descriptor of the (windowed) row matrix in box_rows-row boxes, cached on the handle until the rows move,
// grow or the box changes.
int row_tmap(ivr_index* idx, int box_rows, const CUtensorMap** tmx);
// Queries to fp16 [nq_pad, dpad] with their scales and -inf thresholds, bracketed by the prep timing marks, then
// their TMA descriptor in box_rows-row boxes.  `zero_bytes` at `zero` are cleared inside the bracket.
int prepare_queries(ivr_index* idx, bool timed, const float* q_dev, int64_t nq, int64_t nq_pad, __half* q_h,
                    float* q_scale, uint32_t* tau_g, int box_rows, CUtensorMap* tmq, cudaStream_t st,
                    void* zero = nullptr, size_t zero_bytes = 0);

// A batch searched in n seeded launches: after each scoring launch, fold_launch(seq, ph, lists) merges its candidate
// lists -- straight into D / I when n == 1, otherwise into per-launch keys whose exact k-th best score per query
// raises the shared thresholds (tau_g) of the next launch; finish_launches merges the per-launch keys into D / I.
// The caller marks kScoreBegin before the first scoring launch; the scoring launches are bracketed together, so with
// several launches the (tiny) merges between them count as score_ms.
struct LaunchSeq {
    ivr_index*   idx;
    cudaStream_t st;
    bool         timed;
    int64_t      nq;
    int          k, n;                       // n = number of launches
    float*       D;
    int64_t*     I;
    int64_t      id_offset;
    // workspace: fp16 queries [nq_pad, dpad], their scales and thresholds [nq_pad], per-launch keys [n][nq][k] and
    // counts [n][nq], merge scratch for up to max_lists lists per query, then the caller's own part
    __half*   q_h;
    float*    q_scale;
    uint32_t* tau_g;
    uint64_t* keys, *tmp_e;
    int*      counts, *tmp_c;
    char*     own;
};
// Lays out the workspace of a sequence whose first nine fields are set, with own_bytes for the caller at seq->own.
int begin_launches(LaunchSeq* seq, int64_t nq_pad, int max_lists, size_t own_bytes);
int fold_launch(LaunchSeq& seq, int ph, const MergeIn& lists);
int finish_launches(LaunchSeq& seq);

// small-batch kernel (search_mma_small.cu)
int  search_mma_small(ivr_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev,
                      int64_t id_offset, cudaStream_t st);
// its range epilogue: one launch of <= small_range_chunk() queries that appends every (row, query) with
// score > radius to the hit pool of range_search.cu; with `cut`, only over the row tiles and rows of that part of a
// selection (search_mma_small_sel_range_kernel)
int  search_mma_small_range(ivr_index* idx, const __half* q_h, const float* q_scale, int64_t nq, int64_t q_base,
                            float radius, unsigned long long* cursor, uint64_t* keys, uint32_t* qidx, int64_t capacity,
                            cudaStream_t st, const SelCut* cut = nullptr);
// its self-join epilogue: one launch that appends both (i, j) and (j, i) of every pair i < j of the stored rows with
// score > radius to the hit pool of range_search.cu
int  search_mma_small_join(ivr_index* idx, float radius, unsigned long long* cursor, uint64_t* keys, uint32_t* qidx,
                           int64_t capacity, cudaStream_t st);
// its cross-join epilogue: every pair (stored row i, other row j) with score > radius, two pool entries each, keys of
// global ids (self_id0 + i, other_id0 + j), segments i and n + j; one launch per 2^31-1 work units
int  search_mma_small_cross_join(ivr_index* idx, const __half* other, int64_t n_other, bool other_is_lower,
                                 uint32_t self_id0, uint32_t other_id0, float radius, unsigned long long* cursor,
                                 uint64_t* keys, uint32_t* qidx, int64_t capacity, cudaStream_t st);

}  // namespace ivr

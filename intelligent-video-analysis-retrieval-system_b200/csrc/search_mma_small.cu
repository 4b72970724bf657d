// search_mma_small.cu -- K1s: the tcgen05 search for SMALL query batches (2 .. 128 queries).
//
// With a handful of queries the search is bound by streaming the rows from HBM once (SURVEY.md 8d:
// N * D * 2 bytes per batch).  The batched kernels of search_mma.cu put the QUERIES on the UMMA M
// axis, so 16 queries still cost a full M = 256 instruction per 256 rows -- profiling showed the
// tensor pipe 82 % busy (and the SM clock power-capped) multiplying padding, and 70-75 % of the HBM
// rate.  Here the operands are swapped:
//
//     D[rows (M = 128 TMEM lanes), queries (N = npad columns)] = X_tile[128, dpad] * Q[npad, dpad]^T
//
// so the tensor work is proportional to the number of queries (N = 16 .. 128) and the kernel is a
// pure row streamer:
//   * the query matrix (npad x dpad fp16, <= 128 KB) is loaded ONCE per CTA and stays in shared memory;
//   * warp 0 (one lane) streams 128-row tiles through a TMA/mbarrier ring of 16 KB stages
//     (one 64-column k-block of 128 rows each, SWIZZLE_128B), every CTA a contiguous range of tiles;
//   * warp 1 (one lane) issues tcgen05.mma cta_group::1 kind::f16 (M = 128, N = npad, K = 16) into one
//     of up to 8 TMEM accumulators of npad columns;
//   * warps 2-5 drain the accumulators: tcgen05.ld hands every THREAD one ROW's scores for 32 queries;
//     each is compared with its query's admission threshold (shared memory, refreshed from the
//     per-query threshold all CTAs share through global memory); survivors are appended with a warp
//     ballot to the (CTA, warp, query) candidate list; a list that could overflow on the next tile is
//     compacted to its k best by a warp bitonic sort (registers for k <= 128, in memory above), which
//     also raises the thresholds.
// Large shards are searched in up to three launches of growing size (one tile per CTA, then ~380x
// more, then the rest): the exact k-th best of the rows seen so far seeds the thresholds of the
// next launch, so that lists almost never need compaction (the cold start of 4 x 148 lists per
// query would otherwise cost more than the streaming itself).
// The per-(CTA, warp) survivors are folded by topk_merge.cu.
// A third epilogue, with a fixed threshold, runs in its own __global__ (search_mma_small_range_kernel) for the exact
// range search of range_search.cu; it shares the producer and MMA code below.  A fourth, search_mma_small_join_kernel,
// serves the self-join of range_search.cu: stored rows on both operands, the upper triangle of the score matrix.  A
// fifth, search_mma_small_cross_join_kernel, scores the whole rectangle of two different row sets (one rank's window
// against another rank's rows in ShardedFlatIP.range_self_join).
// Filtered search (ivr_selection, selection.cu) runs the top-k and range epilogues in their own __global__ functions,
// search_mma_small_sel_kernel and search_mma_small_sel_range_kernel: the producer streams the row tiles of the
// selection's tile list, and each epilogue warp ANDs its 32 rows' bitmap word into the row-validity test.  The kernel
// bodies are templates on the row-tile source (AllRows / SelRows), so the unfiltered kernels compile as before.
// A filtered search under a search window streams the UNSHIFTED stored rows: the host cuts the window's tiles out of
// the selection's list, p.n_rows ends the window and SelRows::row_lo starts it (windows need not be tile-aligned).
//
// Replaces D, I = index.search(x, k) for small batches (unified_index.py:503, core.py:891).
// Algorithmic bytes: ntotal * dpad * 2 per search.
#include "mma_common.cuh"

#include <climits>
#include <numeric>

namespace ivr {

constexpr int kSmallThreads    = 192;                  // producer, MMA issuer, 4 epilogue warps
constexpr int kSmallTileRows   = 128;                  // rows per tile (UMMA M)
constexpr int kSmallStageBytes = kSmallTileRows * 128; // one k-block of a row tile: 16 KB
constexpr size_t kSmallMaxListBytes = 2ull << 30;      // candidate-list workspace bound (large k x many queries)
constexpr int kSmallMaxQ       = 128;                  // queries per launch (UMMA N)
constexpr int kSmallMaxBuf     = 8;                    // TMEM accumulators
constexpr int kSmallAuxBytes   = 4096;                 // barriers + thresholds + per-warp counts

struct SmallParams {
    int64_t n_rows;          // rows in this shard
    int     nq, npad;        // real queries; padded to a multiple of 16 (UMMA N)
    int     k;
    int     C;               // candidate list capacity: 2 * kcap(k) (256 for k <= 128: register sort)
    int     kblocks;         // dpad / 64
    int     stages;          // row ring depth (16 KB each)
    int     nbuf, buf_cols;  // TMEM accumulators and their column stride
    int64_t nt;              // row tiles of this launch
    int64_t tile0;           // first row tile of this launch (row id = (tile0 + j) * 128 + lane)
    uint64_t row_policy;     // L2 eviction priority of the row loads
    uint64_t* lists;         // [grid][4 warps][npad][C] raw candidate lists
    int*      counts;        // [grid][4 warps][npad]
    uint32_t* tau_g;         // [npad] shared per-query thresholds (order-preserving encoding)
    // DUMP mode (small shards: dump != nullptr): no candidate lists -- every score goes to dump[q * dump_stride + row]
    // (4 bytes per (query, row): a few % of the row bytes for the batches this kernel serves) and every 128-row tile
    // publishes its maximum per query, tile_max[q * n_tiles + tile]; merge_select_kernel then needs only the ~k tiles
    // whose maximum reaches the k-th largest tile maximum.  One launch, no threshold learning, no seeding launches.
    float*    dump;
    int64_t   dump_stride;   // floats per query (>= padded row count)
    uint32_t* tile_max;      // zero-initialised by the caller
    int64_t   n_tiles;       // tiles of the whole shard
    uint32_t* group_max;     // [npad][n_groups]: maxima of n_groups runs of consecutive tiles (zero-initialised)
    int       n_groups;
};

__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}

// Shared-memory layout of every K1s kernel: [query tile | row ring | aux]; aux holds the mbarriers, the TMEM address
// slot and (from byte 512) the per-query thresholds.
struct SmallSmem {
    uint8_t* gen_base;              // generic address of smem_q
    uint32_t smem_q, smem_a, aux;
    uint32_t q_block, q_bytes;      // one k-block of the query matrix; all of it
    __device__ __forceinline__ SmallSmem(uint8_t* smem_raw, int npad, int kblocks, int stages) {
        smem_q = (smem_u32(smem_raw) + 1023u) & ~1023u;
        gen_base = smem_raw + (smem_q - smem_u32(smem_raw));
        q_block = static_cast<uint32_t>(npad) * 128u;
        q_bytes = kblocks * q_block;
        smem_a = smem_q + q_bytes;
        aux = smem_a + stages * kSmallStageBytes;
    }
    __device__ __forceinline__ uint32_t full_bar(int s) const   { return aux + 8u * s; }
    __device__ __forceinline__ uint32_t empty_bar(int s) const  { return aux + 8u * (16 + s); }
    __device__ __forceinline__ uint32_t q_full() const          { return aux + 8u * 32; }
    __device__ __forceinline__ uint32_t tfull_bar(int a) const  { return aux + 8u * (34 + a); }
    __device__ __forceinline__ uint32_t tempty_bar(int a) const { return aux + 8u * (42 + a); }
    __device__ __forceinline__ uint32_t tmem_slot() const       { return aux + 8u * 50; }
    __device__ __forceinline__ float* tau_s() const { return reinterpret_cast<float*>(gen_base + (aux - smem_q) + 512); }
};

// Prologue shared by the K1s kernels, before their __syncthreads: barriers, descriptor prefetch, TMEM allocation.
__device__ __forceinline__ void small_setup(const SmallSmem& sm, const CUtensorMap* tmap_q, const CUtensorMap* tmap_x,
                                            int stages, int nbuf, int warp, int lane) {
    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) { mbar_init(sm.full_bar(s), 1); mbar_init(sm.empty_bar(s), 1); }
        mbar_init(sm.q_full(), 1);
        for (int a = 0; a < nbuf; ++a) { mbar_init(sm.tfull_bar(a), 1); mbar_init(sm.tempty_bar(a), 4); }
        fence_barrier_init();
    }
    if (warp == 0 && lane == 0) { tma_prefetch_desc(tmap_q); tma_prefetch_desc(tmap_x); }
    if (warp == 1) tmem_alloc<1>(sm.tmem_slot(), 512);
}

// Which row tiles a launch streams and which of their rows it may report.  The unfiltered kernels stream the
// consecutive tiles tile0 + j and report every row; the filtered ones (search_mma_small_sel*_kernel) stream tile
// tiles[j] of a selection's tile list and report the rows at or above row_lo whose bit is set in its bitmap: bit lane of
// word tile * 4 + quarter is row tile * 128 + quarter * 32 + lane, the 32 rows one epilogue warp drains.  row_lo is the
// first row of a search window (0 without one); the window's end is SmallParams::n_rows.
struct AllRows {
    int64_t tile0;
    __device__ __forceinline__ int64_t tile(int64_t j) const { return tile0 + j; }
    __device__ __forceinline__ bool selected(int64_t, int, int) const { return true; }
    __device__ __forceinline__ bool dump(const SmallParams& p) const { return p.dump != nullptr; }
};
struct SelRows {
    const uint32_t* tiles;             // ascending tile ids; position j of the launch is tiles[j]
    const uint32_t* words;             // the row bitmap, zero-padded to whole tiles
    int64_t         row_lo;            // rows below it are not reported
    __device__ __forceinline__ int64_t tile(int64_t j) const { return __ldg(tiles + j); }
    __device__ __forceinline__ bool selected(int64_t t, int quarter, int lane) const {
        return t * kSmallTileRows + quarter * 32 + lane >= row_lo && ((__ldg(words + t * 4 + quarter) >> lane) & 1u);
    }
    __device__ __forceinline__ bool dump(const SmallParams&) const { return false; }
};

// Warp 0, one lane: the query tile once, then row tiles rows.tile(j), j in [j0, j1), through the ring.
template <class Rows>
__device__ __forceinline__ void small_produce(const SmallSmem& sm, const CUtensorMap* tmap_q, const CUtensorMap* tmap_x,
                                              int kblocks, int stages, const Rows& rows, int64_t j0, int64_t j1,
                                              uint64_t row_policy) {
    mbar_expect_tx(sm.q_full(), sm.q_bytes);
    for (int kb = 0; kb < kblocks; ++kb)
        tma_load_2d<1>(sm.smem_q + kb * sm.q_block, tmap_q, sm.q_full(), kb * kKBlock, 0, kL2EvictLast);
    int stage = 0; uint32_t phase = 0;
    for (int64_t j = j0; j < j1; ++j) {
        const int row0 = static_cast<int>(rows.tile(j) * kSmallTileRows);
        for (int kb = 0; kb < kblocks; ++kb) {
            mbar_wait(sm.empty_bar(stage), phase ^ 1);
            mbar_expect_tx(sm.full_bar(stage), kSmallStageBytes);
            tma_load_2d<1>(sm.smem_a + stage * kSmallStageBytes, tmap_x, sm.full_bar(stage), kb * kKBlock, row0, row_policy);
            if (++stage == stages) { stage = 0; phase ^= 1; }
        }
    }
}

// Warp 1, one lane: D[128 rows, npad queries] of each row tile into the next of the nbuf TMEM accumulators.
__device__ __forceinline__ void small_mma(const SmallSmem& sm, uint32_t tmem_base, int npad, int kblocks, int stages,
                                          int nbuf, int buf_cols, int64_t j0, int64_t j1) {
    const uint32_t idesc = make_idesc(kSmallTileRows, npad);
    mbar_wait(sm.q_full(), 0);
    tc_fence_after();
    int stage = 0; uint32_t phase = 0; int buf = 0; uint32_t bphase = 0;
    for (int64_t j = j0; j < j1; ++j) {
        mbar_wait(sm.tempty_bar(buf), bphase ^ 1);                  // epilogue drained this accumulator
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(buf * buf_cols);
        for (int kb = 0; kb < kblocks; ++kb) {
            mbar_wait(sm.full_bar(stage), phase);
            tc_fence_after();
            const uint32_t a0 = sm.smem_a + stage * kSmallStageBytes;   // A: streamed rows (M)
            const uint32_t b0 = sm.smem_q + kb * sm.q_block;            // B: resident queries (N)
#pragma unroll
            for (int k4 = 0; k4 < kKBlock / 16; ++k4)
                umma_f16<1>(tmem_d, make_smem_desc(a0 + k4 * 32), make_smem_desc(b0 + k4 * 32), idesc,
                            (kb | k4) ? 1u : 0u);
            umma_commit<1>(sm.empty_bar(stage));                    // ring slot free when these MMAs retire
            if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        umma_commit<1>(sm.tfull_bar(buf));
        if (++buf == nbuf) { buf = 0; bphase ^= 1; }
    }
}

// The body of the top-k kernels: the candidate-list epilogue over row tiles rows.tile(j), j in [j0, j1) -- and, for the
// unfiltered kernel, dump mode (SmallParams::dump).
template <class Rows>
__device__ __forceinline__ void small_topk(const CUtensorMap& tmap_q, const CUtensorMap& tmap_x, const SmallParams& p,
                                           const Rows& rows) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const SmallSmem sm(smem_raw, p.npad, p.kblocks, p.stages);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* const tau_s = sm.tau_s();                                                          // [128]
    int*   const cnt_s = reinterpret_cast<int*>(sm.gen_base + (sm.aux - sm.smem_q) + 1024);   // [4][128]

    const int64_t j0 = p.nt * blockIdx.x / gridDim.x, j1 = p.nt * (blockIdx.x + 1) / gridDim.x;   // owned row tiles

    small_setup(sm, &tmap_q, &tmap_x, p.stages, p.nbuf, warp, lane);
    for (int i = threadIdx.x; i < 4 * kSmallMaxQ; i += kSmallThreads) cnt_s[i] = 0;
    for (int i = threadIdx.x; i < kSmallMaxQ; i += kSmallThreads)      // padded queries admit nothing
        tau_s[i] = (i < p.nq) ? ord2f(__ldcg(p.tau_g + i)) : __int_as_float(0x7f800000);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(sm.tmem_slot()));

    if (warp == 0 && lane == 0) {
        small_produce(sm, &tmap_q, &tmap_x, p.kblocks, p.stages, rows, j0, j1, p.row_policy);
    } else if (warp == 1 && lane == 0) {
        small_mma(sm, tmem_base, p.npad, p.kblocks, p.stages, p.nbuf, p.buf_cols, j0, j1);
    } else if (warp >= 2) {
        // ============================ epilogue: fused top-k ====================
        const int quarter = warp & 3;                              // the TMEM lanes this warp may read
        int* const cnt_w = cnt_s + quarter * kSmallMaxQ;
        const int64_t wslot = static_cast<int64_t>(blockIdx.x) * 4 + quarter;
        uint64_t* const wl = p.lists + wslot * p.npad * p.C;
        const unsigned lt_mask = (1u << lane) - 1u;

        auto compact = [&](int q) {                                // all lanes; list of query q
            const int c = cnt_w[q];
            __syncwarp();
            uint64_t* const lst = wl + static_cast<int64_t>(q) * p.C;
            const float t = (p.C == 256) ? warp_compact_raw<8>(lst, c, p.k, p.C, lane)      // register bitonic sort
                                         : warp_compact_raw<0>(lst, c, p.k, p.C, lane);     // in-memory (k > 128)
            if (lane == 0) {
                cnt_w[q] = min(c, p.k);
                if (c >= p.k) {
                    if (t > tau_s[q]) tau_s[q] = t;                // benign race: any value is a valid lower bound
                    atomicMax(p.tau_g + q, f2ord(t));              // share with the other CTAs
                }
            }
            __syncwarp();
        };

        int buf = 0; uint32_t bphase = 0; int64_t n = 0;
        if (rows.dump(p)) {
            // ---------------- dump mode: scores + per-tile maxima, no lists ----------------
            for (int64_t j = j0; j < j1; ++j) {
                const int64_t tile = p.tile0 + j;
                const int64_t grp = tile * p.n_groups / p.n_tiles;
                const int64_t row = tile * kSmallTileRows + quarter * 32 + lane;
                const bool valid = row < p.n_rows;
                mbar_wait(sm.tfull_bar(buf), bphase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                                       static_cast<uint32_t>(buf * p.buf_cols);
                for (int c0 = 0; c0 < p.npad; c0 += 32) {
                    uint32_t v[32];
                    const int ncol = min(32, p.npad - c0);
                    if (ncol == 32) tmem_ld_32x32(taddr + c0, v);
                    else tmem_ld_32x16(taddr + c0, v);                  // npad is a multiple of 16
                    tmem_wait_ld(v);
                    if (c0 + 32 >= p.npad) {                            // accumulator fully read: hand it back
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_local(sm.tempty_bar(buf));
                    }
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        if (i >= ncol) break;                           // warp-uniform
                        const uint32_t bits = valid ? v[i] : 0xff800000u;   // rows past the end: -inf
                        float* dst = p.dump + static_cast<int64_t>(c0 + i) * p.dump_stride + row;
                        *dst = __uint_as_float(bits);                    // 32 consecutive rows: one 128-byte store per query
                        // the maxima bound the scores the merge keys, which skips NaN: a NaN counts as -inf here
                        const uint32_t mb = (bits & 0x7fffffffu) > 0x7f800000u ? 0xff800000u : bits;
                        const uint32_t mx = __reduce_max_sync(0xffffffffu, f2ord(__uint_as_float(mb)));
                        if (lane == 0) {
                            atomicMax(p.tile_max + static_cast<int64_t>(c0 + i) * p.n_tiles + tile, mx);
                            atomicMax(p.group_max + static_cast<int64_t>(c0 + i) * p.n_groups + grp, mx);
                        }
                    }
                }
                if (++buf == p.nbuf) { buf = 0; bphase ^= 1; }
            }
        } else
        for (int64_t j = j0; j < j1; ++j, ++n) {
            // make room: one tile adds at most 32 entries (one per lane) to each of this warp's lists
            for (int qb = 0; qb < p.npad; qb += 32) {
                const int q = qb + lane;
                unsigned need = __ballot_sync(0xffffffffu, q < p.npad && cnt_w[q] > p.C - 32);
                while (need) { const int l = __ffs(need) - 1; need &= need - 1; compact(qb + l); }
            }
            // fold in the thresholds the other CTAs have published (one warp per tile, round robin)
            if (static_cast<int>(n & 3) == quarter)
                for (int q = lane; q < p.nq; q += 32) {
                    const float t = ord2f(__ldcg(p.tau_g + q));
                    if (t > tau_s[q]) tau_s[q] = t;
                }
            __syncwarp();
            const int64_t tile = rows.tile(j);
            const uint32_t row = static_cast<uint32_t>(tile * kSmallTileRows + quarter * 32 + lane);
            const bool valid = static_cast<int64_t>(row) < p.n_rows && rows.selected(tile, quarter, lane);
            mbar_wait(sm.tfull_bar(buf), bphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                                   static_cast<uint32_t>(buf * p.buf_cols);
            for (int c0 = 0; c0 < p.npad; c0 += 32) {
                uint32_t v[32];
                if (p.npad - c0 >= 32) {
                    tmem_ld_32x32(taddr + c0, v);
                } else {                                            // npad is a multiple of 16: a 16-column tail
#pragma unroll
                    for (int i = 16; i < 32; ++i) v[i] = 0xff800000u;
                    tmem_ld_32x16(taddr + c0, v);
                }
                tmem_wait_ld(v);
                if (c0 + 32 >= p.npad) {                            // accumulator fully read: hand it back
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(sm.tempty_bar(buf));
                }
                unsigned m = 0;
                const float4* t4 = reinterpret_cast<const float4*>(tau_s + c0);
#pragma unroll
                for (int i4 = 0; i4 < 8; ++i4) {
                    const float4 t = t4[i4];
                    m |= (__uint_as_float(v[4 * i4 + 0]) > t.x ? 1u : 0u) << (4 * i4 + 0);
                    m |= (__uint_as_float(v[4 * i4 + 1]) > t.y ? 1u : 0u) << (4 * i4 + 1);
                    m |= (__uint_as_float(v[4 * i4 + 2]) > t.z ? 1u : 0u) << (4 * i4 + 2);
                    m |= (__uint_as_float(v[4 * i4 + 3]) > t.w ? 1u : 0u) << (4 * i4 + 3);
                }
                if (!valid) m = 0;                                  // rows past the end of the shard (TMA zero fill)
                const unsigned wm = __reduce_or_sync(0xffffffffu, m);
                if (wm == 0) continue;
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    if (!(wm & (1u << i))) continue;                // warp-uniform
                    const bool hit = (m >> i) & 1u;
                    const unsigned hits = __ballot_sync(0xffffffffu, hit);
                    const int q = c0 + i;
                    const int base = cnt_w[q];
                    if (hit)
                        wl[static_cast<int64_t>(q) * p.C + base + __popc(hits & lt_mask)] =
                            static_cast<uint64_t>(v[i]) | (static_cast<uint64_t>(row) << 32);
                    __syncwarp();
                    if (lane == 0) cnt_w[q] = base + __popc(hits);
                }
                __syncwarp();
            }
            if (++buf == p.nbuf) { buf = 0; bphase ^= 1; }
        }
        __syncwarp();
        if (!rows.dump(p))
            for (int q = lane; q < p.npad; q += 32) p.counts[wslot * p.npad + q] = cnt_w[q];
    }

    // ------------------------------------------------------------------ teardown ----
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<1>(tmem_base, 512);
}

__global__ void __launch_bounds__(kSmallThreads, 1)
search_mma_small_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x,
                        const SmallParams p) {
    small_topk(tmap_q, tmap_x, p, AllRows{p.tile0});
}

// Filtered top-k: the list epilogue over the row tiles of a selection (SelRows).  p.tile0 and p.nt count positions in
// the selection's tile list, so the seeded launches split the list as the unfiltered ones split the rows.  Rows below
// row_lo or at or past p.n_rows are never reported.  No dump mode.
__global__ void __launch_bounds__(kSmallThreads, 1)
search_mma_small_sel_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x,
                            const SmallParams p, const uint32_t* __restrict__ tiles, const uint32_t* __restrict__ words,
                            int64_t row_lo) {
    small_topk(tmap_q, tmap_x, p, SelRows{tiles + p.tile0, words, row_lo});
}

// The largest fp32 t with fp32(t * scale) <= radius, so that "score > t" is exactly "the reported score, fp32(score *
// scale), > radius".  scale is a power of two, so this is radius / scale whenever that division is exact; at the ends
// of the float range the rescaled scores round (to subnormals or to inf) and the threshold moves to the rounding
// boundary of radius instead: mid, between radius and the next float up, rounds to whichever is even.
__device__ __forceinline__ float range_threshold(float radius, float scale) {
    if (isinf(radius) && radius > 0.f) return radius;
    const float up = nextafterf(radius, __int_as_float(0x7f800000));
    const double mid = 0.5 * (static_cast<double>(radius) + (isinf(up) ? 0x1p128 : static_cast<double>(up)));
    const double b = mid / static_cast<double>(scale);
    float t = __double2float_rd(b);
    if ((__float_as_uint(radius) & 1u) && static_cast<double>(t) == b) t = nextafterf(t, __int_as_float(0xff800000));
    return t;
}

// RANGE mode: the same producer and MMA warps; the epilogue compares every score with a threshold that never moves
// (range_threshold(radius, q_scale[q])) and appends the survivors to ONE hit pool shared by all CTAs and launches.  One
// 64-bit cursor reservation per warp and 32-query chunk, no lists, no compaction, no counts.  Writes at or past
// `capacity` are dropped, but the cursor still advances, so the true total is always known.
struct SmallRangeParams {
    int64_t  n_rows;
    int      nq, npad, kblocks, stages, nbuf, buf_cols;
    int64_t  nt;                       // row tiles (the whole index: one launch per query chunk)
    uint64_t row_policy;
    float        radius;
    const float* q_scale;              // [nq] power-of-two query scales of this launch
    uint32_t     q_base;               // global index of this launch's first query
    unsigned long long* cursor;        // hits reserved so far, by every launch of the search
    uint64_t*    keys;                 // [capacity] make_key(score in the kernel's domain, row)
    uint32_t*    qidx;                 // [capacity] global query index of each key
    unsigned long long capacity;
};

// The body of the range kernels: the fixed-threshold epilogue over row tiles rows.tile(j), j in [j0, j1).
template <class Rows>
__device__ __forceinline__ void small_range(const CUtensorMap& tmap_q, const CUtensorMap& tmap_x, const SmallRangeParams& p,
                                            const Rows& rows) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const SmallSmem sm(smem_raw, p.npad, p.kblocks, p.stages);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* const tau_s = sm.tau_s();                                   // [128]
    const int64_t j0 = p.nt * blockIdx.x / gridDim.x, j1 = p.nt * (blockIdx.x + 1) / gridDim.x;

    small_setup(sm, &tmap_q, &tmap_x, p.stages, p.nbuf, warp, lane);
    for (int i = threadIdx.x; i < kSmallMaxQ; i += kSmallThreads)      // padded queries admit nothing
        tau_s[i] = (i < p.nq) ? range_threshold(p.radius, p.q_scale[i]) : __int_as_float(0x7f800000);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(sm.tmem_slot()));

    if (warp == 0 && lane == 0) {
        small_produce(sm, &tmap_q, &tmap_x, p.kblocks, p.stages, rows, j0, j1, p.row_policy);
    } else if (warp == 1 && lane == 0) {
        small_mma(sm, tmem_base, p.npad, p.kblocks, p.stages, p.nbuf, p.buf_cols, j0, j1);
    } else if (warp >= 2) {
        // ============================ epilogue: fixed-threshold filter ========
        const int quarter = warp & 3;                              // the TMEM lanes this warp may read
        int buf = 0; uint32_t bphase = 0;
        for (int64_t j = j0; j < j1; ++j) {
            const int64_t tile = rows.tile(j);
            const int64_t row64 = tile * kSmallTileRows + quarter * 32 + lane;
            const bool valid = row64 < p.n_rows && rows.selected(tile, quarter, lane);
            const uint32_t row = static_cast<uint32_t>(row64);
            mbar_wait(sm.tfull_bar(buf), bphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                                   static_cast<uint32_t>(buf * p.buf_cols);
            for (int c0 = 0; c0 < p.npad; c0 += 32) {
                uint32_t v[32];
                if (p.npad - c0 >= 32) {
                    tmem_ld_32x32(taddr + c0, v);
                } else {                                            // npad is a multiple of 16: a 16-column tail
#pragma unroll
                    for (int i = 16; i < 32; ++i) v[i] = 0xff800000u;
                    tmem_ld_32x16(taddr + c0, v);
                }
                tmem_wait_ld(v);
                if (c0 + 32 >= p.npad) {                            // accumulator fully read: hand it back
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(sm.tempty_bar(buf));
                }
                unsigned m = 0;
                const float4* t4 = reinterpret_cast<const float4*>(tau_s + c0);
#pragma unroll
                for (int i4 = 0; i4 < 8; ++i4) {
                    const float4 t = t4[i4];
                    m |= (__uint_as_float(v[4 * i4 + 0]) > t.x ? 1u : 0u) << (4 * i4 + 0);
                    m |= (__uint_as_float(v[4 * i4 + 1]) > t.y ? 1u : 0u) << (4 * i4 + 1);
                    m |= (__uint_as_float(v[4 * i4 + 2]) > t.z ? 1u : 0u) << (4 * i4 + 2);
                    m |= (__uint_as_float(v[4 * i4 + 3]) > t.w ? 1u : 0u) << (4 * i4 + 3);
                }
                if (!valid) m = 0;                                  // rows past the end (TMA zero fill)
                // one reservation for the warp's hits, each lane's slots from an inclusive prefix sum
                const int cnt = __popc(m);
                int incl = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += t;
                }
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                if (total == 0) continue;                           // warp-uniform
                unsigned long long slot = 0;
                if (lane == 0) slot = atomicAdd(p.cursor, static_cast<unsigned long long>(total));
                slot = __shfl_sync(0xffffffffu, slot, 0) + static_cast<unsigned long long>(incl - cnt);
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    if (!((m >> i) & 1u)) continue;
                    if (slot < p.capacity) {
                        p.keys[slot] = make_key(__uint_as_float(v[i]), row);
                        p.qidx[slot] = p.q_base + static_cast<uint32_t>(c0 + i);
                    }
                    ++slot;
                }
            }
            if (++buf == p.nbuf) { buf = 0; bphase ^= 1; }
        }
    }

    // ------------------------------------------------------------------ teardown ----
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<1>(tmem_base, 512);
}

__global__ void __launch_bounds__(kSmallThreads, 1)
search_mma_small_range_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x,
                              const SmallRangeParams p) {
    small_range(tmap_q, tmap_x, p, AllRows{0});
}

// Filtered range search: the fixed-threshold epilogue over the row tiles of a selection (SelRows); p.nt counts
// positions in the selection's tile list; rows below row_lo or at or past p.n_rows are never reported.
__global__ void __launch_bounds__(kSmallThreads, 1)
search_mma_small_sel_range_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x,
                                  const SmallRangeParams p, const uint32_t* __restrict__ tiles,
                                  const uint32_t* __restrict__ words, int64_t row_lo) {
    small_range(tmap_q, tmap_x, p, SelRows{tiles, words, row_lo});
}

// JOIN mode (range_self_join of range_search.cu): both operands are stored rows.  A unit of work is (column block b,
// segment s): B = the npad rows [b * npad, (b + 1) * npad) resident in shared memory, A = the row tiles
// [s * seg_tiles, (s + 1) * seg_tiles) that hold a row below the block's last row.  Units are numbered segment-major,
// so the CTAs resident together stream the same row tiles and L2 serves all but the first read of each.  seg_tiles *
// 128 is a multiple of npad: segment s starts at block s * seg_blocks and holds nb - s * seg_blocks units.
struct SmallJoinParams {
    int64_t  n;                        // rows of the (windowed) index
    int      npad, kblocks, stages, nbuf, buf_cols;
    int      seg_tiles;                // row tiles per segment
    int64_t  nb, seg_blocks, n_seg;    // column blocks; blocks a segment start moves by; segments
    uint64_t row_policy;
    float    radius;
    unsigned long long* cursor;        // pool entries reserved so far
    uint64_t* keys;                    // [capacity] make_key(score, column row)
    uint32_t* qidx;                    // [capacity] the other row of the pair
    unsigned long long capacity;
};

// Warp 0, one lane: the npad-row block of B at row b_row once, then row tiles [t0, t1) of A through the ring.
__device__ __forceinline__ void small_produce_join(const SmallSmem& sm, const CUtensorMap* tmap_b, int b_row,
                                                   const CUtensorMap* tmap_x, int kblocks, int stages, int64_t t0,
                                                   int64_t t1, uint64_t policy) {
    mbar_expect_tx(sm.q_full(), sm.q_bytes);
    for (int kb = 0; kb < kblocks; ++kb)
        tma_load_2d<1>(sm.smem_q + kb * sm.q_block, tmap_b, sm.q_full(), kb * kKBlock, b_row, policy);
    int stage = 0; uint32_t phase = 0;
    for (int64_t t = t0; t < t1; ++t) {
        const int row0 = static_cast<int>(t * kSmallTileRows);
        for (int kb = 0; kb < kblocks; ++kb) {
            mbar_wait(sm.empty_bar(stage), phase ^ 1);
            mbar_expect_tx(sm.full_bar(stage), kSmallStageBytes);
            tma_load_2d<1>(sm.smem_a + stage * kSmallStageBytes, tmap_x, sm.full_bar(stage), kb * kKBlock, row0, policy);
            if (++stage == stages) { stage = 0; phase ^= 1; }
        }
    }
}

// One CTA per unit (see SmallJoinParams).  The epilogue keeps (i, j) with i < j < n and score > radius and appends
// two pool entries per pair, (make_key(s, j), i) and (make_key(s, i), j): one 64-bit cursor reservation per warp and
// 32-column chunk.  Entries at or past `capacity` are dropped but counted.
__global__ void __launch_bounds__(kSmallThreads, 1)
search_mma_small_join_kernel(const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_x,
                             const SmallJoinParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const SmallSmem sm(smem_raw, p.npad, p.kblocks, p.stages);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // unit -> (segment s, block b): segments before s hold P(s) = s * nb - seg_blocks * s * (s - 1) / 2 units
    const int64_t u = blockIdx.x;
    int64_t lo = 0, hi = p.n_seg - 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (mid * p.nb - p.seg_blocks * mid * (mid - 1) / 2 <= u) lo = mid; else hi = mid - 1;
    }
    const int64_t s = lo;
    const int64_t b = s * p.seg_blocks + (u - (s * p.nb - p.seg_blocks * s * (s - 1) / 2));
    const int64_t jb = b * p.npad;                                     // first column row
    const int64_t j_end = jb + p.npad < p.n ? jb + p.npad : p.n;
    const int64_t t_end = (j_end + kSmallTileRows - 1) / kSmallTileRows;   // the tiles up to the block's last row
    const int64_t t0 = s * p.seg_tiles, t1 = t0 + p.seg_tiles < t_end ? t0 + p.seg_tiles : t_end;

    small_setup(sm, &tmap_b, &tmap_x, p.stages, p.nbuf, warp, lane);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(sm.tmem_slot()));

    if (warp == 0 && lane == 0) {
        small_produce_join(sm, &tmap_b, static_cast<int>(jb), &tmap_x, p.kblocks, p.stages, t0, t1, p.row_policy);
    } else if (warp == 1 && lane == 0) {
        small_mma(sm, tmem_base, p.npad, p.kblocks, p.stages, p.nbuf, p.buf_cols, t0, t1);
    } else if (warp >= 2) {
        // ============================ epilogue: upper triangle, fixed threshold ========
        const int quarter = warp & 3;                              // the TMEM lanes this warp may read
        int buf = 0; uint32_t bphase = 0;
        for (int64_t t = t0; t < t1; ++t) {
            const int64_t i = t * kSmallTileRows + quarter * 32 + lane;
            mbar_wait(sm.tfull_bar(buf), bphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                                   static_cast<uint32_t>(buf * p.buf_cols);
            for (int c0 = 0; c0 < p.npad; c0 += 32) {
                uint32_t v[32];
                if (p.npad - c0 >= 32) {
                    tmem_ld_32x32(taddr + c0, v);
                } else {                                            // npad is a multiple of 16: a 16-column tail
#pragma unroll
                    for (int k = 16; k < 32; ++k) v[k] = 0xff800000u;
                    tmem_ld_32x16(taddr + c0, v);
                }
                tmem_wait_ld(v);
                if (c0 + 32 >= p.npad) {                            // accumulator fully read: hand it back
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(sm.tempty_bar(buf));
                }
                unsigned m = 0;
#pragma unroll
                for (int k = 0; k < 32; ++k) m |= (__uint_as_float(v[k]) > p.radius ? 1u : 0u) << k;
                // column k is row j = jc + k: keep i < j < n.  This also drops the zero-filled rows past n, whose
                // score 0 can exceed a negative radius, and every A row i >= n (then no j > i is below n).
                const int64_t jc = jb + c0;
                const int64_t above = i - jc, below = p.n - jc;     // keep k > above and k < below
                m &= above < 0 ? 0xffffffffu : (above >= 31 ? 0u : 0xffffffffu << (above + 1));
                m &= below >= 32 ? 0xffffffffu : (below <= 0 ? 0u : (1u << below) - 1u);
                const int cnt = __popc(m);
                int incl = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int x = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += x;
                }
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                if (total == 0) continue;                           // warp-uniform
                unsigned long long slot = 0;
                if (lane == 0) slot = atomicAdd(p.cursor, 2ull * static_cast<unsigned long long>(total));
                slot = __shfl_sync(0xffffffffu, slot, 0) + 2ull * static_cast<unsigned long long>(incl - cnt);
                const uint32_t row_i = static_cast<uint32_t>(i);
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    if (!((m >> k) & 1u)) continue;
                    const float sc = __uint_as_float(v[k]);
                    const uint32_t row_j = static_cast<uint32_t>(jc + k);
                    if (slot < p.capacity)     { p.keys[slot] = make_key(sc, row_j);     p.qidx[slot] = row_i; }
                    if (slot + 1 < p.capacity) { p.keys[slot + 1] = make_key(sc, row_i); p.qidx[slot + 1] = row_j; }
                    slot += 2;
                }
            }
            if (++buf == p.nbuf) { buf = 0; bphase ^= 1; }
        }
    }

    // ------------------------------------------------------------------ teardown ----
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<1>(tmem_base, 512);
}

// CROSS-JOIN mode (range_cross_join_keys_device of range_search.cu): two different row sets, A (the one with the lower
// global ids, streamed in 128-row tiles) and B (npad-row blocks resident in shared memory).  Every pair (i in A, j in
// B) is scored, so a unit is (column block b, segment s) of the full rectangle; units are numbered segment-major,
// u = s * nb + b, and a launch covers units [u0, u0 + gridDim.x).  Row ids in the pool are global: A row i is
// a_id0 + i and lands in segment a_seg0 + i, B row j likewise.
struct SmallCrossParams {
    int64_t  n_a, n_b;                 // rows of A and of B
    int      npad, kblocks, stages, nbuf, buf_cols;
    int      seg_tiles;                // row tiles of A per segment
    int64_t  nb;                       // column blocks of B
    int64_t  u0;                       // first unit of this launch
    uint64_t row_policy;
    float    radius;
    uint32_t a_id0, b_id0;             // global id of row 0 of A / of B
    uint32_t a_seg0, b_seg0;           // pool segment of row 0 of A / of B
    unsigned long long* cursor;        // pool entries reserved so far
    uint64_t* keys;                    // [capacity] make_key(score, global id of the partner)
    uint32_t* qidx;                    // [capacity] the segment of the row the entry belongs to
    unsigned long long capacity;
};

// One CTA per unit.  The epilogue keeps (i, j) with i < n_a, j < n_b and score > radius -- the bounds are explicit
// because the zero-filled rows past either end score 0, which exceeds a negative radius -- and appends two pool entries
// per pair, one for each row, from one 64-bit cursor reservation per warp and 32-column chunk.  Entries at or past
// `capacity` are dropped but counted.
__global__ void __launch_bounds__(kSmallThreads, 1)
search_mma_small_cross_join_kernel(const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_a,
                                   const SmallCrossParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const SmallSmem sm(smem_raw, p.npad, p.kblocks, p.stages);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    const int64_t u = p.u0 + blockIdx.x;
    const int64_t s = u / p.nb, b = u - s * p.nb;
    const int64_t jb = b * p.npad;                                     // first B row of the block
    const int64_t t_end = (p.n_a + kSmallTileRows - 1) / kSmallTileRows;
    const int64_t t0 = s * p.seg_tiles, t1 = t0 + p.seg_tiles < t_end ? t0 + p.seg_tiles : t_end;

    small_setup(sm, &tmap_b, &tmap_a, p.stages, p.nbuf, warp, lane);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(sm.tmem_slot()));

    if (warp == 0 && lane == 0) {
        small_produce_join(sm, &tmap_b, static_cast<int>(jb), &tmap_a, p.kblocks, p.stages, t0, t1, p.row_policy);
    } else if (warp == 1 && lane == 0) {
        small_mma(sm, tmem_base, p.npad, p.kblocks, p.stages, p.nbuf, p.buf_cols, t0, t1);
    } else if (warp >= 2) {
        // ============================ epilogue: the rectangle, fixed threshold ========
        const int quarter = warp & 3;                              // the TMEM lanes this warp may read
        int buf = 0; uint32_t bphase = 0;
        for (int64_t t = t0; t < t1; ++t) {
            const int64_t i = t * kSmallTileRows + quarter * 32 + lane;
            mbar_wait(sm.tfull_bar(buf), bphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                                   static_cast<uint32_t>(buf * p.buf_cols);
            for (int c0 = 0; c0 < p.npad; c0 += 32) {
                uint32_t v[32];
                if (p.npad - c0 >= 32) {
                    tmem_ld_32x32(taddr + c0, v);
                } else {                                            // npad is a multiple of 16: a 16-column tail
#pragma unroll
                    for (int k = 16; k < 32; ++k) v[k] = 0xff800000u;
                    tmem_ld_32x16(taddr + c0, v);
                }
                tmem_wait_ld(v);
                if (c0 + 32 >= p.npad) {                            // accumulator fully read: hand it back
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(sm.tempty_bar(buf));
                }
                unsigned m = 0;
#pragma unroll
                for (int k = 0; k < 32; ++k) m |= (__uint_as_float(v[k]) > p.radius ? 1u : 0u) << k;
                // column k is B row j = jc + k: keep i < n_a and j < n_b
                const int64_t jc = jb + c0;
                const int64_t below = p.n_b - jc;                   // keep k < below
                if (i >= p.n_a) m = 0;
                m &= below >= 32 ? 0xffffffffu : (below <= 0 ? 0u : (1u << below) - 1u);
                const int cnt = __popc(m);
                int incl = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int x = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += x;
                }
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                if (total == 0) continue;                           // warp-uniform
                unsigned long long slot = 0;
                if (lane == 0) slot = atomicAdd(p.cursor, 2ull * static_cast<unsigned long long>(total));
                slot = __shfl_sync(0xffffffffu, slot, 0) + 2ull * static_cast<unsigned long long>(incl - cnt);
                const uint32_t id_i = p.a_id0 + static_cast<uint32_t>(i), seg_i = p.a_seg0 + static_cast<uint32_t>(i);
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    if (!((m >> k) & 1u)) continue;
                    const float sc = __uint_as_float(v[k]);
                    const uint32_t j = static_cast<uint32_t>(jc + k);
                    if (slot < p.capacity)     { p.keys[slot] = make_key(sc, p.b_id0 + j); p.qidx[slot] = seg_i; }
                    if (slot + 1 < p.capacity) { p.keys[slot + 1] = make_key(sc, id_i); p.qidx[slot + 1] = p.b_seg0 + j; }
                    slot += 2;
                }
            }
            if (++buf == p.nbuf) { buf = 0; bphase ^= 1; }
        }
    }

    // ------------------------------------------------------------------ teardown ----
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<1>(tmem_base, 512);
}

// ------------------------------------------------------------------ host side ----
struct SmallShape { int npad, stages, nbuf, buf_cols, C; size_t smem; };

// Pipeline shape of a K1s launch over nq queries: false when the resident query tile does not fit.
static bool pipe_shape(const ivr_index* idx, int64_t nq, SmallShape* s) {
    if (nq < 1 || nq > kSmallMaxQ) return false;
    const int npad = static_cast<int>((nq + 15) / 16 * 16);
    const int64_t q_bytes = static_cast<int64_t>(npad) * idx->dpad * 2;
    if (q_bytes > 128 * 1024) return false;
    const int stages = std::min<int64_t>(12, (kSmemBudget - 1024 - kSmallAuxBytes - q_bytes) / kSmallStageBytes);
    if (stages < 4) return false;
    s->npad = npad; s->stages = stages; s->C = 0;
    s->buf_cols = std::max(npad, 32);
    s->nbuf = std::min(kSmallMaxBuf, 512 / s->buf_cols);
    s->smem = 1024 + static_cast<size_t>(q_bytes) + static_cast<size_t>(stages) * kSmallStageBytes + kSmallAuxBytes;
    return true;
}

static bool small_shape(const ivr_index* idx, int64_t nq, int k, SmallShape* s) {
    if (k < 1 || k > IVR_MAX_K || !pipe_shape(idx, nq, s)) return false;
    const int C = 2 * kcap_for(k);
    if (static_cast<size_t>(4 * idx->sm_count) * s->npad * C * 8 > kSmallMaxListBytes) return false;   // huge k x many queries
    s->C = C;
    return true;
}

bool mma_small_supported(const ivr_index* idx, int64_t nq, int k) {
    SmallShape s;
    return small_shape(idx, nq, k, &s);
}

// One launch in dump mode + the one-launch select (merge_select_kernel, dense input).
static int search_mma_small_dump(ivr_index* idx, const SmallShape& sh, const float* q_dev, int64_t nq, int k, float* D_dev,
                                 int64_t* I_dev, int64_t id_offset, cudaStream_t st) {
    const int64_t nt = (idx->ntotal + kSmallTileRows - 1) / kSmallTileRows;
    const int64_t stride = nt * kSmallTileRows;                      // padded rows per query
    Carve carve;
    const size_t o_q  = carve(static_cast<size_t>(sh.npad) * idx->dpad * 2);
    const size_t o_sc = carve(static_cast<size_t>(sh.npad) * 4);
    const size_t o_tg = carve(static_cast<size_t>(sh.npad) * 4);
    const size_t o_s  = carve(static_cast<size_t>(sh.npad) * stride * 4);
    const int n_groups = static_cast<int>(std::min<int64_t>(nt, 1024));
    const size_t zero_bytes = (static_cast<size_t>(sh.npad) * (nt + n_groups) + 2 * nq) * 4;   // tile + group maxima, pool counters, tickets
    const size_t o_z  = carve(zero_bytes);
    const size_t o_p  = carve(static_cast<size_t>(nq) * kSelectPoolCap * 8);
    IVR_TRY(ensure_ws(idx, carve.size));
    char* ws = static_cast<char*>(idx->ws);
    __half* q_h = reinterpret_cast<__half*>(ws + o_q);
    float* q_scale = reinterpret_cast<float*>(ws + o_sc);
    uint32_t* tau_g = reinterpret_cast<uint32_t*>(ws + o_tg);
    uint32_t* tile_max = reinterpret_cast<uint32_t*>(ws + o_z);
    uint32_t* group_max = tile_max + static_cast<size_t>(sh.npad) * nt;
    int* pool_cnt = reinterpret_cast<int*>(group_max + static_cast<size_t>(sh.npad) * n_groups);
    const bool timed = idx->timing;

    CUtensorMap tmq;
    const CUtensorMap* tmx;
    IVR_TRY(prepare_queries(idx, timed, q_dev, nq, sh.npad, q_h, q_scale, tau_g, sh.npad, &tmq, st, ws + o_z, zero_bytes));
    IVR_TRY(row_tmap(idx, kSmallTileRows, &tmx));
    IVR_CUDA(cudaFuncSetAttribute(search_mma_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(sh.smem)));
    SmallParams p{};
    p.n_rows = idx->ntotal; p.nq = static_cast<int>(nq); p.npad = sh.npad; p.k = k; p.C = sh.C;
    p.kblocks = idx->dpad / kKBlock; p.stages = sh.stages; p.nbuf = sh.nbuf; p.buf_cols = sh.buf_cols;
    p.tile0 = 0; p.nt = nt;
    p.row_policy = kL2EvictFirst;
    p.tau_g = tau_g;
    p.dump = reinterpret_cast<float*>(ws + o_s); p.dump_stride = stride; p.tile_max = tile_max; p.n_tiles = nt;
    p.group_max = group_max; p.n_groups = n_groups;
    const int grid = static_cast<int>(std::min<int64_t>(idx->sm_count, std::max<int64_t>(nt, 1)));
    timing_mark(idx, timed, kScoreBegin, st);
    search_mma_small_kernel<<<grid, kSmallThreads, sh.smem, st>>>(tmq, *tmx, p);
    IVR_CUDA(cudaGetLastError());
    idx->launches[0]++;
    timing_mark(idx, timed, kScoreEnd, st); timing_mark(idx, timed, kMergeBegin, st);
    MergeIn in{};
    in.dense = p.dump; in.dense_q_stride = stride; in.dense_rows = idx->ntotal; in.dense_len = kSmallTileRows;
    in.cnt_list_stride = 1; in.cnt_q_stride = nt;                   // strides of the maxima array
    in.n_lists = static_cast<int>(nt);
    IVR_TRY(merge_select_final(in, tile_max, nq, k, D_dev, I_dev, id_offset, reinterpret_cast<uint64_t*>(ws + o_p),
                               pool_cnt, pool_cnt + nq, idx->sm_count, st, &idx->launches[1], q_scale, group_max, n_groups));
    timing_mark(idx, timed, kMergeEnd, st);
    if (timed) idx->ev_valid[0] = idx->ev_valid[1] = idx->ev_valid[2] = true;
    idx->last_kernel = "search_mma_small_kernel";
    return IVR_OK;
}

// The seeded candidate-list launches over nt row tiles (for the filtered kernel: positions in a selection's tile list),
// merged into D / I (packed keys into I when D == nullptr); rows at or past n_rows are not reported.
// launch(grid, tmq, tmx, p) queues one scoring launch of `kernel`.  time_first marks the query preparation and the start
// of the scoring, time_last the end of the scoring and the final merge.
template <class Launch>
static int small_list_search(ivr_index* idx, const SmallShape& sh, const float* q_dev, int64_t nq, int k, float* D_dev,
                             int64_t* I_dev, int64_t id_offset, cudaStream_t st, int64_t nt, int64_t n_rows,
                             const void* kernel, bool time_first, bool time_last, Launch&& launch) {
    const int sms = idx->sm_count;
    // launch boundaries (in row tiles): one tile per CTA, then as many rows as keep the expected admissions per
    // list around 64 (k * rows_now / rows_before spread over 4 * sms lists), then the rest
    int64_t bounds[4] = {0, 0, 0, 0};
    int n_phases = 1;
    if (env_int("IVR_MMA_TWO_PHASE", 1) && nt >= 4 * static_cast<int64_t>(sms)) {
        const int64_t b0 = sms;
        const int64_t ratio = std::max<int64_t>(2, env_int("IVR_MMA_SMALL_RATIO", 0) > 0 ? env_int("IVR_MMA_SMALL_RATIO", 0)
                                                                                     : static_cast<int64_t>(sh.C / 4) * 4 * sms / k);
        const int64_t b1 = b0 + b0 * ratio;
        bounds[n_phases++] = b0;
        if (nt > b1 + b1 / 2) bounds[n_phases++] = b1;
    }
    bounds[n_phases] = nt;

    const int max_grid = static_cast<int>(std::min<int64_t>(sms, std::max<int64_t>(nt, 1)));
    const int max_lists = std::max(4 * max_grid, 3);
    Carve own;
    const size_t o_l = own(static_cast<size_t>(max_lists) * sh.npad * sh.C * 8);
    const size_t o_c = own(static_cast<size_t>(max_lists) * sh.npad * 4);
    LaunchSeq seq{idx, st, time_last, nq, k, n_phases, D_dev, I_dev, id_offset};
    IVR_TRY(begin_launches(&seq, sh.npad, max_lists, own.size));

    CUtensorMap tmq;
    const CUtensorMap* tmx;
    IVR_TRY(prepare_queries(idx, time_first, q_dev, nq, sh.npad, seq.q_h, seq.q_scale, seq.tau_g, sh.npad, &tmq, st));
    IVR_TRY(row_tmap(idx, kSmallTileRows, &tmx));
    IVR_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sh.smem)));

    timing_mark(idx, time_first, kScoreBegin, st);
    for (int ph = 0; ph < n_phases; ++ph) {
        SmallParams p{};
        p.n_rows = n_rows; p.nq = static_cast<int>(nq); p.npad = sh.npad; p.k = k; p.C = sh.C;
        p.kblocks = idx->dpad / kKBlock; p.stages = sh.stages; p.nbuf = sh.nbuf; p.buf_cols = sh.buf_cols;
        p.tile0 = bounds[ph]; p.nt = bounds[ph + 1] - bounds[ph];
        p.row_policy = kL2EvictFirst;                                // every row is read exactly once
        p.lists = reinterpret_cast<uint64_t*>(seq.own + o_l);
        p.counts = reinterpret_cast<int*>(seq.own + o_c);
        p.tau_g = seq.tau_g;
        const int grid = static_cast<int>(std::min<int64_t>(sms, std::max<int64_t>(p.nt, 1)));
        launch(grid, tmq, *tmx, p);
        IVR_CUDA(cudaGetLastError());
        idx->launches[0]++;
        MergeIn in{};
        in.entries = p.lists; in.counts = p.counts;
        in.list_stride = static_cast<int64_t>(sh.npad) * sh.C; in.q_stride = sh.C;
        in.cnt_list_stride = sh.npad; in.cnt_q_stride = 1;
        in.n_lists = 4 * grid; in.fixed_count = 0; in.raw = 1;
        IVR_TRY(fold_launch(seq, ph, in));
    }
    return finish_launches(seq);
}

int search_mma_small(ivr_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev,
                     int64_t id_offset, cudaStream_t st) {
    SmallShape sh;
    if (!small_shape(idx, nq, k, &sh)) { set_error("search_mma_small: unsupported shape (nq=%lld, k=%d, dim=%d)",
                                                   static_cast<long long>(nq), k, idx->dim); return IVR_EUNSUPPORTED; }
    const int64_t nt = (idx->ntotal + kSmallTileRows - 1) / kSmallTileRows;
    // Small shards: one launch that materialises the scores (see SmallParams::dump).  The seeded candidate-list path
    // pays ~0.2 ms of fixed cost (2-3 launches, their merges, cold lists); writing the scores costs nq * 4 bytes per
    // row.  Measured (dump vs lists, ms): 1 M x 512: 16 q 0.26 vs 0.37, 32 q 0.30 vs 0.37, 64 q 0.44 vs 0.41;
    // 851 k x 768: 16 q 0.30 vs 0.41, 64 q 0.37 vs 0.43; 3 M x 512: 16 q 0.64 vs 0.68, 32 q 0.72 vs 0.68; 4 M: equal;
    // 6 M: lists win.  Rule: up to 3.5 M rows while the scores add at most 1/6 to the row bytes.
    // IVR_SMALL_DUMP_MAX_KROWS (0 = never) overrides the row limit: tests use it to reach both modes.
    const int64_t dump_rows = static_cast<int64_t>(env_int("IVR_SMALL_DUMP_MAX_KROWS", 3500)) * 1000;
    if (k <= kSelectMaxK && idx->ntotal <= dump_rows && sh.npad * 4 * 6 <= idx->dpad * 2)
        return search_mma_small_dump(idx, sh, q_dev, nq, k, D_dev, I_dev, id_offset, st);
    IVR_TRY(small_list_search(idx, sh, q_dev, nq, k, D_dev, I_dev, id_offset, st, nt, idx->ntotal,
                              reinterpret_cast<const void*>(search_mma_small_kernel), idx->timing, idx->timing,
                              [&](int grid, const CUtensorMap& tmq, const CUtensorMap& tmx, const SmallParams& p) {
        search_mma_small_kernel<<<grid, kSmallThreads, sh.smem, st>>>(tmq, tmx, p);
    }));
    idx->last_kernel = "search_mma_small_kernel";
    return IVR_OK;
}

int small_sel_chunk(const ivr_index* idx, int k) {
    SmallShape sh;
    for (int c = kSmallMaxQ; c >= 16; c -= 16)
        if (small_shape(idx, c, k, &sh)) return c;
    return 0;
}

int search_mma_small_selected(ivr_index* idx, const SelCut& cut, const float* q_dev, int64_t nq, int k, float* D_dev,
                              int64_t* I_dev, int64_t id_offset, cudaStream_t st) {
    const int chunk = small_sel_chunk(idx, k);
    if (chunk == 0) {
        set_error("search_selected: dim %d with k=%d does not fit the small-batch kernel", idx->dim, k);
        return IVR_EUNSUPPORTED;
    }
    const int64_t n_chunks = (nq + chunk - 1) / chunk;
    for (int64_t c = 0; c < n_chunks; ++c) {
        const int64_t q0 = c * chunk, m = std::min<int64_t>(chunk, nq - q0);
        SmallShape sh;
        small_shape(idx, m, k, &sh);                                 // fits: m <= chunk
        IVR_TRY(small_list_search(idx, sh, q_dev + q0 * idx->dim, m, k, D_dev ? D_dev + q0 * k : nullptr,
                                  I_dev + q0 * k, id_offset, st, cut.n_tiles, cut.row_hi,
                                  reinterpret_cast<const void*>(search_mma_small_sel_kernel),
                                  idx->timing && c == 0, idx->timing && c == n_chunks - 1,
                                  [&](int grid, const CUtensorMap& tmq, const CUtensorMap& tmx, const SmallParams& p) {
            search_mma_small_sel_kernel<<<grid, kSmallThreads, sh.smem, st>>>(tmq, tmx, p, cut.tiles, cut.words,
                                                                              cut.row_lo);
        }));
    }
    idx->last_kernel = "search_mma_small_sel_kernel";
    return IVR_OK;
}

int small_range_chunk(const ivr_index* idx) {
    return std::min(kSmallMaxQ, 65536 / idx->dpad / 16 * 16);
}

int search_mma_small_range(ivr_index* idx, const __half* q_h, const float* q_scale, int64_t nq, int64_t q_base,
                           float radius, unsigned long long* cursor, uint64_t* keys, uint32_t* qidx, int64_t capacity,
                           cudaStream_t st, const SelCut* cut) {
    SmallShape sh;
    if (nq > small_range_chunk(idx) || !pipe_shape(idx, nq, &sh)) {
        set_error("range_search: %lld queries of dim %d do not fit one query tile", static_cast<long long>(nq), idx->dim);
        return IVR_EUNSUPPORTED;
    }
    CUtensorMap tmq;
    const CUtensorMap* tmx;
    IVR_TRY(make_tmap(&tmq, q_h, sh.npad, idx->dpad, sh.npad));
    IVR_TRY(row_tmap(idx, kSmallTileRows, &tmx));
    const void* kernel = cut ? reinterpret_cast<const void*>(search_mma_small_sel_range_kernel)
                             : reinterpret_cast<const void*>(search_mma_small_range_kernel);
    IVR_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sh.smem)));
    SmallRangeParams p{};
    p.n_rows = cut ? cut->row_hi : idx->ntotal; p.nq = static_cast<int>(nq); p.npad = sh.npad;
    p.kblocks = idx->dpad / kKBlock; p.stages = sh.stages; p.nbuf = sh.nbuf; p.buf_cols = sh.buf_cols;
    p.nt = cut ? cut->n_tiles : (idx->ntotal + kSmallTileRows - 1) / kSmallTileRows;
    p.row_policy = kL2EvictFirst;                                    // each launch reads every row once
    p.radius = radius; p.q_scale = q_scale; p.q_base = static_cast<uint32_t>(q_base);
    p.cursor = cursor; p.keys = keys; p.qidx = qidx; p.capacity = static_cast<unsigned long long>(capacity);
    const int grid = static_cast<int>(std::min<int64_t>(idx->sm_count, std::max<int64_t>(p.nt, 1)));
    if (cut) search_mma_small_sel_range_kernel<<<grid, kSmallThreads, sh.smem, st>>>(tmq, *tmx, p, cut->tiles, cut->words,
                                                                                    cut->row_lo);
    else search_mma_small_range_kernel<<<grid, kSmallThreads, sh.smem, st>>>(tmq, *tmx, p);
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

// One CTA per unit rather than a persistent grid: a CTA then never reloads B behind MMAs still reading it, and the
// units, ~40 row tiles of 1.8 us of tensor work each at 512 dims, are long enough that the set-up of a CTA (barriers,
// TMEM, the 128 KB block of B) costs a few percent.
int search_mma_small_join(ivr_index* idx, float radius, unsigned long long* cursor, uint64_t* keys, uint32_t* qidx,
                          int64_t capacity, cudaStream_t st) {
    const int64_t n = idx->ntotal;
    const int npad = small_range_chunk(idx);
    SmallShape sh;
    if (!pipe_shape(idx, npad, &sh)) {
        set_error("range_self_join: dim %d does not fit the small-batch kernel", idx->dim);
        return IVR_EUNSUPPORTED;
    }
    int seg_tiles = npad / std::gcd(npad, kSmallTileRows);          // the least tile count that ends on a block edge
    seg_tiles *= (40 + seg_tiles - 1) / seg_tiles;                  // ~40 row tiles per unit
    SmallJoinParams p{};
    p.n = n; p.npad = sh.npad;
    p.kblocks = idx->dpad / kKBlock; p.stages = sh.stages; p.nbuf = sh.nbuf; p.buf_cols = sh.buf_cols;
    p.seg_tiles = seg_tiles;
    p.nb = (n + npad - 1) / npad;
    p.seg_blocks = static_cast<int64_t>(seg_tiles) * kSmallTileRows / npad;
    p.n_seg = ((n + kSmallTileRows - 1) / kSmallTileRows + seg_tiles - 1) / seg_tiles;
    const int64_t units = p.n_seg * p.nb - p.seg_blocks * p.n_seg * (p.n_seg - 1) / 2;
    if (units > INT_MAX) {
        set_error("range_self_join: %lld rows need %lld work units, more than one launch holds (2^31-1)",
                  static_cast<long long>(n), static_cast<long long>(units));
        return IVR_EUNSUPPORTED;
    }
    p.row_policy = kL2EvictNormal;                                   // other CTAs re-read the same row tiles
    p.radius = radius;
    p.cursor = cursor; p.keys = keys; p.qidx = qidx; p.capacity = static_cast<unsigned long long>(capacity);
    const CUtensorMap* cached;
    IVR_TRY(row_tmap(idx, kSmallTileRows, &cached));
    const CUtensorMap tmx = *cached;                                 // the cache holds one box height at a time
    IVR_TRY(row_tmap(idx, npad, &cached));
    const CUtensorMap tmb = *cached;
    IVR_CUDA(cudaFuncSetAttribute(search_mma_small_join_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(sh.smem)));
    search_mma_small_join_kernel<<<static_cast<unsigned>(units), kSmallThreads, sh.smem, st>>>(tmb, tmx, p);
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

// The rectangle of the (windowed) index rows against `other` ([n_other, dpad] fp16 on the index's device).  The set
// with the lower global ids is A, as i is in the self-join, so a pair's score has the bits the single-index join gives
// it.  More units than one launch holds (2^31-1; IVR_JOIN_MAX_UNITS lowers the limit) are split into launches over
// consecutive unit ranges.
int search_mma_small_cross_join(ivr_index* idx, const __half* other, int64_t n_other, bool other_is_lower,
                                uint32_t self_id0, uint32_t other_id0, float radius, unsigned long long* cursor,
                                uint64_t* keys, uint32_t* qidx, int64_t capacity, cudaStream_t st) {
    const int64_t n_self = idx->ntotal;
    const int npad = small_range_chunk(idx);
    SmallShape sh;
    if (!pipe_shape(idx, npad, &sh)) {
        set_error("range_cross_join: dim %d does not fit the small-batch kernel", idx->dim);
        return IVR_EUNSUPPORTED;
    }
    SmallCrossParams p{};
    p.n_a = other_is_lower ? n_other : n_self;
    p.n_b = other_is_lower ? n_self : n_other;
    p.npad = sh.npad;
    p.kblocks = idx->dpad / kKBlock; p.stages = sh.stages; p.nbuf = sh.nbuf; p.buf_cols = sh.buf_cols;
    p.seg_tiles = 40;                                                // ~40 row tiles per unit, as in the self-join
    p.nb = (p.n_b + npad - 1) / npad;
    p.row_policy = kL2EvictNormal;                                   // other CTAs re-read the same row tiles
    p.radius = radius;
    p.a_id0 = other_is_lower ? other_id0 : self_id0;
    p.b_id0 = other_is_lower ? self_id0 : other_id0;
    p.a_seg0 = other_is_lower ? static_cast<uint32_t>(n_self) : 0u;
    p.b_seg0 = other_is_lower ? 0u : static_cast<uint32_t>(n_self);
    p.cursor = cursor; p.keys = keys; p.qidx = qidx; p.capacity = static_cast<unsigned long long>(capacity);
    const int64_t n_seg = ((p.n_a + kSmallTileRows - 1) / kSmallTileRows + p.seg_tiles - 1) / p.seg_tiles;
    const int64_t units = n_seg * p.nb;
    if (units == 0) return IVR_OK;
    const CUtensorMap* cached;
    IVR_TRY(row_tmap(idx, other_is_lower ? npad : kSmallTileRows, &cached));
    const CUtensorMap tmi = *cached;
    CUtensorMap tmo;
    IVR_TRY(make_tmap(&tmo, other, n_other, idx->dpad, other_is_lower ? kSmallTileRows : npad));
    const CUtensorMap& tma = other_is_lower ? tmo : tmi;
    const CUtensorMap& tmb = other_is_lower ? tmi : tmo;
    IVR_CUDA(cudaFuncSetAttribute(search_mma_small_cross_join_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(sh.smem)));
    const int64_t max_units = std::max<int64_t>(1, std::min<int64_t>(INT_MAX, env_int("IVR_JOIN_MAX_UNITS", INT_MAX)));
    for (int64_t u0 = 0; u0 < units; u0 += max_units) {
        p.u0 = u0;
        const int64_t grid = std::min(max_units, units - u0);
        search_mma_small_cross_join_kernel<<<static_cast<unsigned>(grid), kSmallThreads, sh.smem, st>>>(tmb, tma, p);
        IVR_CUDA(cudaGetLastError());
    }
    return IVR_OK;
}

}  // namespace ivr

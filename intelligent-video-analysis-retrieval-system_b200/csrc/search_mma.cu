// search_mma.cu -- K1+K2: batched exact search on the 5th-gen tensor cores.
//
// Replaces D, I = index.search(x, k) for query batches (unified_index.py:503 is
// called once per query by the reference; core.py:891 already passes [nq, d]).
//
//   S[q, r] = <Q[q,:], X[r,:]>      Q: [nq, dpad] fp16 (converted + pow2-scaled per call)
//                                   X: [ntotal, dpad] fp16 rows, HBM resident
//
// One persistent CTA per SM (CG = 1) or one CTA pair per TPC (CG = 2,
// tcgen05 cta_group::2).  A work unit is a (128*CG queries) x (256 rows) tile.
//   * SCHEDULE.  With G CTA groups and Tq query tiles, c = floor(G / Tq) groups are bound to every
//     query tile for the whole kernel (the "grid" part, c * Tq groups): group (t, i) owns query
//     tile t and walks the row tiles i, i + c, i + 2c, ... -- so at any moment all Tq query tiles
//     are working on the same c row tiles: the first group to touch a row tile fetches it from
//     HBM, the other Tq - 1 hit it in L2 (measured: without this lockstep every query tile
//     re-read the rows from HBM).  The G - c * Tq leftover groups take the last
//     (G - c*Tq)/G of the row tiles, query-tile-major, so every group has the same MMA work.
//   * the query tile stays RESIDENT in shared memory (dpad <= 512: 128 x dpad fp16
//     = 128 KB) -- only the row tiles stream through a TMA/mbarrier ring, which
//     halves the L2->SMEM traffic of a classic GEMM tile loop;
//   * warp 0 (one lane) issues TMA loads (cp.async.bulk.tensor, SWIZZLE_128B);
//   * warp 1 (one lane) issues tcgen05.mma kind::f16 (fp16 x fp16 -> fp32) into one
//     of two 256-column TMEM accumulators;
//   * warps 4-11 are two epilogue sets, one per accumulator: tcgen05.ld hands every
//     THREAD one query's 32 scores per instruction; the thread compares them with that
//     query's admission threshold (register; the max of its own k-th best and a
//     per-query threshold shared by all CTAs through global memory), a warp vote skips
//     chunks without survivors, survivors are appended branch-free (predicated stores)
//     to the query's candidate list; the 32 interleaved lists of a warp are pruned together, lane-parallel
//     (warp_prune_lists in mma_common.cuh), when one of them nears its capacity.
//     The score matrix never reaches shared or global memory.
// The raw per-(slot, set, query) lists are folded by topk_merge.cu.  A search runs as a few launches of growing
// size; each one's exact k-th best scores seed the admission thresholds of the next (search_mma_batch).
//
// Algorithmic work: 2 * ntotal * dpad * nq FLOP per search (SURVEY.md 8d).
#include "mma_common.cuh"

#include <cmath>

// Pipeline probes (epilogue skipped / tcgen05.ld only) return garbage results: they exist only in builds made
// with -DIVR_PROBES (tools/probe_epilogue.sh) and are compiled out of the shipped library.
#ifdef IVR_PROBES
#define IVR_SKIP_EPI(p) ((p).skip_epilogue)
#else
#define IVR_SKIP_EPI(p) 0
#endif

namespace ivr {


// One 32-column chunk of one query's scores (v) against its admission threshold; survivors go to the
// thread's candidate list (entry i at my_list[i * 32]: the lists of a warp are interleaved).  Sub-maxima of
// the four 8-column groups are formed with independent 3-input max trees (short dependency
// chains); a warp vote per group skips groups without survivors, so the common "one survivor in
// the whole warp-chunk" case costs 8 predicated stores instead of 32.
__device__ __forceinline__ void filter_chunk(const uint32_t (&v)[32], float tau, int& cnt, uint64_t* my_list,
                                             uint32_t rowc, int col0, int nvalid, int tile_rows = kTileN) {
    float g8[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        const float a = fmaxf(fmaxf(__uint_as_float(v[8 * g]), __uint_as_float(v[8 * g + 1])), __uint_as_float(v[8 * g + 2]));
        const float b = fmaxf(fmaxf(__uint_as_float(v[8 * g + 3]), __uint_as_float(v[8 * g + 4])), __uint_as_float(v[8 * g + 5]));
        g8[g] = fmaxf(fmaxf(a, b), fmaxf(__uint_as_float(v[8 * g + 6]), __uint_as_float(v[8 * g + 7])));
    }
    const float m = fmaxf(fmaxf(g8[0], g8[1]), fmaxf(g8[2], g8[3]));
    if (!__any_sync(0xffffffffu, m > tau)) return;
    if (nvalid == tile_rows) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            if (!__any_sync(0xffffffffu, g8[g] > tau)) continue;       // warp-uniform
#pragma unroll
            for (int i = 8 * g; i < 8 * g + 8; ++i) {                  // branch-free: predicated 8-byte store
                const float sc = __uint_as_float(v[i]);
                uint64_t* dst = my_list + static_cast<int64_t>(cnt) * kListStride;
                asm volatile(
                    "{\n\t.reg .pred pp;\n\tsetp.gt.f32 pp, %0, %1;\n\t"
                    "@pp st.global.v2.b32 [%2], {%3, %4};\n\t}"
                    ::"f"(sc), "f"(tau), "l"(dst), "r"(v[i]), "r"(rowc + i) : "memory");
                cnt += (sc > tau) ? 1 : 0;
            }
        }
    } else {                                                            // last, partial row tile of the shard
        for (int i = 0; i < 32; ++i) {
            const float sc = __uint_as_float(v[i]);
            if (sc > tau && col0 + i < nvalid) {
                my_list[static_cast<int64_t>(cnt) * kListStride] = static_cast<uint64_t>(v[i]) | (static_cast<uint64_t>(rowc + i) << 32);
                ++cnt;
            }
        }
    }
}

struct MmaParams {
    int64_t n_rows;          // rows in this shard
    int     nq;              // real queries
    int     k;
    int     C;               // candidate list capacity (2 * kcap)
    int     kblocks;         // dpad / 64
    int     stages;          // row-tile ring depth
    int     tq;              // query tiles
    int64_t nt;              // row tiles of this launch
    int64_t tile0;           // first row tile of this launch (row id = (tile0 + j) * 256 + column)
    int     c;               // grid groups per query tile
    int     g_grid;          // c * tq groups walk rows [0, ntg) in lockstep
    int64_t ntg;             // row tiles of the grid part; the leftover groups own [ntg, nt)
    int     stagger;         // grid part: query tile t starts `stagger * t` steps into its row walk
    int     groups;          // CTA groups in the launch
    int     nq_pad;          // tq * 128 * CG
    int     segs_max;        // max query tiles one group touches
    uint64_t row_policy;     // L2 eviction priority of the row-tile loads
    int      skip_epilogue;  // debug/perf probe: drain nothing (results are garbage)
    uint64_t* lists;         // [slots][nq_pad / 32][C][32] raw candidate lists, interleaved per warp
    int*      counts;        // [slots][nq_pad]
    int2*     state;         // [grid CTAs][segs_max][2 sets][128] {cnt, tau bits} of a parked segment
    uint32_t* tau_g;         // [nq_pad] order-preserving encoding of the shared per-query threshold
};

// The unit enumeration shared by all warp roles.
//   f_visit(s, t, reload, visit)            start of the visit of segment s (query tile t)
//   f_unit(s, t, j, n)                      row tile j; n = running unit counter of this group
//   f_visit_end(s, t, visit, release_q)     end of the visit
// A grid group has one segment (its query tile) and a strided walk over [0, ntg); a leftover group
// walks a contiguous range of the query-tile-major units over the row tiles [ntg, nt).
struct LeftRange {                      // leftover group: units u = t * ntl + jl
    int64_t ub, ue, ntl;
    int t_first, nseg;
    __device__ LeftRange(const MmaParams& p, int group) {
        const int gl = group - p.g_grid, Gl = p.groups - p.g_grid;
        ntl = p.nt - p.ntg;
        const int64_t Ul = static_cast<int64_t>(p.tq) * ntl;
        ub = Ul * gl / Gl; ue = Ul * (gl + 1) / Gl;
        t_first = (ntl > 0) ? static_cast<int>(ub / ntl) : 0;
        nseg = (ue > ub) ? static_cast<int>((ue - 1) / ntl) - t_first + 1 : 0;
    }
};

template <typename FV, typename FU, typename FE>
__device__ __forceinline__ void for_each_unit(const MmaParams& p, int group, FV&& f_visit, FU&& f_unit,
                                              FE&& f_visit_end) {
    if (group < p.g_grid) {
        const int t = group % p.tq, i = group / p.tq;
        if (i >= p.ntg) return;
        f_visit(0, t, true, 0);
        // Query tile t runs `stagger * t` steps ahead (cyclically): the Tq groups that share a row
        // tile request it a step apart instead of in the same instant, so the first request has
        // filled L2 by the time the others arrive.
        const int64_t nsteps = (p.ntg - i + p.c - 1) / p.c;
        int64_t m = (static_cast<int64_t>(p.stagger) * t) % nsteps;
        for (int64_t n = 0; n < nsteps; ++n) {
            f_unit(0, t, i + m * p.c, n);
            if (++m == nsteps) m = 0;
        }
        f_visit_end(0, t, 0, true);
    } else {
        const LeftRange lr(p, group);
        int64_t n = 0;
        for (int s = 0; s < lr.nseg; ++s) {
            const int t = lr.t_first + s;
            const int64_t tb = static_cast<int64_t>(t) * lr.ntl;
            const int64_t j0 = p.ntg + (lr.ub > tb ? lr.ub : tb) - tb;
            const int64_t j1 = p.ntg + (lr.ue < tb + lr.ntl ? lr.ue : tb + lr.ntl) - tb;
            f_visit(s, t, true, s);
            for (int64_t j = j0; j < j1; ++j, ++n) f_unit(s, t, j, n);
            f_visit_end(s, t, s, true);
        }
    }
}

template <int CG, int E>
__global__ void __launch_bounds__(kMmaThreads, 1)
search_mma_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x,
                  const MmaParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // dynamic smem base is only guaranteed 16B aligned: round up to the 1024 B the 128B swizzle needs
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cta_rank = (CG == 2) ? cluster_ctarank() : 0u;
    const int group = blockIdx.x / CG;

    constexpr int kRowsPerCta = kTileN / CG;                    // rows of each tile this CTA loads
    const uint32_t stage_bytes = kRowsPerCta * 128;
    const uint32_t q_bytes = p.kblocks * kQBlockBytes;
    const uint32_t smem_q = smem_base;
    const uint32_t smem_b = smem_q + q_bytes;
    const uint32_t bars = smem_b + p.stages * stage_bytes;      // barrier block
    auto full_bar  = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (16 + s); };
    const uint32_t q_full = bars + 8u * 32, q_empty = bars + 8u * 33;
    auto tfull_bar  = [&](int a) { return bars + 8u * (34 + a); };
    auto tempty_bar = [&](int a) { return bars + 8u * (36 + a); };
    const uint32_t tmem_slot = bars + 8u * 40;

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        mbar_init(q_full, 1); mbar_init(q_empty, 1);
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4 * CG); }
        fence_barrier_init();
    }
    if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmap_q); tma_prefetch_desc(&tmap_x); }
    if (warp == 2) tmem_alloc<CG>(tmem_slot, 512);
    tc_fence_before();
    if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    if (warp == 0 && lane == 0) {
        // ============================ TMA producer ============================
        // At a query-tile switch the first ring-full of row tiles of the new visit is issued BEFORE
        // waiting for the MMAs of the old visit to release the resident query tile, so the ring is
        // already full when the new query tile lands.
        int stage = 0; uint32_t phase = 0; int nload = 0;
        bool pending_q = false; int pending_t = 0; int issued_since = 0;
        auto load_q = [&]() {
            if (nload > 0) mbar_wait(q_empty, (nload - 1) & 1);       // MMAs finished with the old query tile
            if (cta_rank == 0) mbar_expect_tx(q_full, q_bytes * CG);
            for (int kb = 0; kb < p.kblocks; ++kb)
                tma_load_2d<CG>(smem_q + kb * kQBlockBytes, &tmap_q, q_full, kb * kKBlock,
                                pending_t * (kTileQ * CG) + static_cast<int>(cta_rank) * kTileQ, kL2EvictLast);
            ++nload;
            pending_q = false;
        };
        for_each_unit(p, group,
            [&](int, int t, bool reload, int) {
                if (!reload) return;
                pending_q = true; pending_t = t; issued_since = 0;
                if (nload == 0) load_q();                              // very first tile: nothing to overlap
            },
            [&](int, int, int64_t j, int64_t) {
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    if (pending_q && issued_since >= p.stages) load_q();
                    mbar_wait(empty_bar(stage), phase ^ 1);
                    if (cta_rank == 0) mbar_expect_tx(full_bar(stage), stage_bytes * CG);
                    tma_load_2d<CG>(smem_b + stage * stage_bytes, &tmap_x, full_bar(stage), kb * kKBlock,
                                    static_cast<int>((p.tile0 + j) * kTileN) + static_cast<int>(cta_rank) * kRowsPerCta,
                                    p.row_policy);
                    ++issued_since;
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
            },
            [&](int, int, int, bool) { if (pending_q) load_q(); });
        // consumed every q_empty completion but the last, in order: wait for the last one so that no
        // asynchronous arrive can land after the CTA has retired
        if (nload > 0) mbar_wait(q_empty, (nload - 1) & 1);
    } else if (warp == 1 && lane == 0) {
        // ============================ MMA issuer (leader CTA) =================
        // q_empty ("the MMAs reading the query tile have retired") is committed at the end of every visit;
        // the producer consumes the completions in order and waits for the last one before it retires, so
        // no asynchronous arrive can land after the CTA has gone.
        constexpr uint32_t idesc = make_idesc(kTileQ * CG, kTileN);
        int stage = 0; uint32_t phase = 0; int nload = 0;
        for_each_unit(p, group,
            [&](int, int, bool reload, int) {
                if (!reload) return;
                if (cta_rank == 0) mbar_wait(q_full, nload & 1);
                ++nload;
            },
            [&](int, int, int64_t, int64_t n) {
                if (cta_rank != 0) return;
                const int acc = static_cast<int>(n & 1);
                const uint32_t acc_phase = static_cast<uint32_t>((n >> 1) & 1);
                mbar_wait(tempty_bar(acc), acc_phase ^ 1);            // epilogue drained this accumulator
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(acc * kTileN);
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint32_t a0 = smem_q + kb * kQBlockBytes;
                    const uint32_t b0 = smem_b + stage * stage_bytes;
#pragma unroll
                    for (int k4 = 0; k4 < kKBlock / 16; ++k4)          // UMMA K = 16 fp16 = 32 bytes
                        umma_f16<CG>(tmem_d, make_smem_desc(a0 + k4 * 32), make_smem_desc(b0 + k4 * 32), idesc,
                                     (kb | k4) ? 1u : 0u);
                    umma_commit<CG>(empty_bar(stage));                 // ring slot free when these MMAs retire
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
                umma_commit<CG>(tfull_bar(acc));                       // accumulator ready for its epilogue set
            },
            [&](int, int, int, bool release_q) {
                if (release_q && cta_rank == 0) umma_commit<CG>(q_empty);
            });
    } else if (warp >= 4) {
        // ============================ epilogue: fused top-k ====================
        const int set = (warp - 4) >> 2;                           // accumulator / list set 0 or 1
        const int quarter = warp & 3;                              // TMEM lanes [32*quarter, +32)
        const int r = quarter * 32 + lane;                         // query row inside this CTA's tile
        const float NEG_INF = __int_as_float(0xff800000), POS_INF = __int_as_float(0x7f800000);
        auto state_ptr = [&](int s) {
            return p.state + ((static_cast<int64_t>(blockIdx.x) * p.segs_max + s) * 2 + set) * kTileQ + r;
        };
        for (int s = 0; s < p.segs_max; ++s) *state_ptr(s) = make_int2(0, __float_as_int(NEG_INF));
        // list slot of this group for query tile t: the c grid groups first, then the leftover groups that touch t
        auto slot_of = [&](int t) {
            if (group < p.g_grid) return group / p.tq;
            const int Gl = p.groups - p.g_grid;
            const int64_t ntl = p.nt - p.ntg, Ul = static_cast<int64_t>(p.tq) * ntl;
            const int glmin = static_cast<int>(((static_cast<int64_t>(t) * ntl + 1) * Gl - 1) / Ul);
            return p.c + (group - p.g_grid - glmin);
        };

        int cnt = 0; float tau = NEG_INF; int64_t q_global = 0; bool q_ok = false;
        uint64_t* my_list = nullptr; int* my_count = nullptr;

        // make room for two more chunks (<= 64 entries): all 32 lists of the warp are pruned together
        auto make_room = [&]() {
            if (!__any_sync(0xffffffffu, cnt > p.C - 64)) return;
            const float tau_before = tau;
            unsigned bad = warp_prune_lists(my_list, cnt, tau, p.k);
            bad |= __ballot_sync(0xffffffffu, cnt > p.C - 64);      // no pivot / no progress (ties): exact compaction
            while (bad) {
                const int l = __ffs(bad) - 1; bad &= bad - 1;
                const int c_l = __shfl_sync(0xffffffffu, cnt, l);
                __syncwarp();
                const float t_l = warp_compact_raw<E>(my_list - lane + l, c_l, p.k, p.C, lane, kListStride);
                if (lane == l) { cnt = min(cnt, p.k); tau = fmaxf(tau, t_l); }
            }
            if (q_ok && tau > tau_before) atomicMax(p.tau_g + q_global, f2ord(tau));   // share with the other CTAs
        };
        auto process_chunk = [&](uint32_t (&v)[32], int c, int64_t row0, int nvalid) {
            if (IVR_SKIP_EPI(p) == 2) return;                        // perf probe: tcgen05.ld traffic only
            filter_chunk(v, tau, cnt, my_list, static_cast<uint32_t>(row0) + c * 32, c * 32, nvalid);
        };

        for_each_unit(p, group,
            [&](int s, int t, bool, int) {                          // visit begin: restore this segment's state
                q_global = static_cast<int64_t>(t) * (kTileQ * CG) + cta_rank * kTileQ + r;
                q_ok = q_global < p.nq;
                const int2 st = *state_ptr(s);
                cnt = st.x;
                tau = q_ok ? __int_as_float(st.y) : POS_INF;        // padded queries admit nothing
                if (q_ok) tau = fmaxf(tau, ord2f(__ldcg(p.tau_g + q_global)));
                const int64_t slot = static_cast<int64_t>(slot_of(t)) * 2 + set;
                my_list = p.lists + (slot * p.nq_pad + (q_global - lane)) * p.C + lane;
                my_count = p.counts + slot * p.nq_pad + q_global;
            },
            [&](int, int, int64_t j, int64_t n) {
                if (static_cast<int>(n & 1) != set) return;
                const uint32_t acc_phase = static_cast<uint32_t>((n >> 1) & 1);
                const int64_t row0 = (p.tile0 + j) * kTileN;
                const int nvalid = static_cast<int>(min(static_cast<int64_t>(kTileN), p.n_rows - row0));
                // the threshold shared by all CTAs: issue the load now, fold it in after this tile
                // (its L2 latency hides behind the chunk loop)
                const uint32_t tg_bits = q_ok ? __ldcg(p.tau_g + q_global) : 0u;
                mbar_wait(tfull_bar(set), acc_phase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                                       static_cast<uint32_t>(set * kTileN);
                uint32_t va[32], vb[32];
                if (IVR_SKIP_EPI(p) != 1) tmem_ld_32x32(taddr, va);
#pragma unroll 1
                for (int c = 0; c < (IVR_SKIP_EPI(p) == 1 ? 0 : kTileN / 32); c += 2) {
                    make_room();
                    tmem_wait_ld(va);
                    tmem_ld_32x32(taddr + (c + 1) * 32, vb);
                    process_chunk(va, c, row0, nvalid);
                    tmem_wait_ld(vb);
                    if (c + 2 < kTileN / 32) tmem_ld_32x32(taddr + (c + 2) * 32, va);
                    process_chunk(vb, c + 1, row0, nvalid);
                }
                if (q_ok) tau = fmaxf(tau, ord2f(tg_bits));
                // every tcgen05.ld of this accumulator has completed: hand it back to the MMA issuer
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if constexpr (CG == 1) mbar_arrive_local(tempty_bar(set));
                    else mbar_arrive_cluster(tempty_bar(set), 0);
                }
            },
            [&](int s, int, int, bool) {                            // visit end: park the state, publish the count
                *state_ptr(s) = make_int2(cnt, __float_as_int(tau));
                *my_count = cnt;                                    // the merge kernel reads the raw list directly
            });
    }

    // ------------------------------------------------------------------ teardown ----
    tc_fence_before();
    if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
    if (warp == 2) tmem_dealloc<CG>(tmem_base, 512);
}


// ===================================================================================
// Row-tile-resident variant (cta_group::2 only), used for large query batches.
//
// Profiling the query-tile-resident kernel at 4096 queries showed the L2 slices 99 % busy and
// every query tile re-fetching the rows from HBM (13x the algorithmic traffic, no schedule --
// phases, lockstep, stagger, eviction hints -- changed that; see profiles/).  Here the roles are
// swapped: a CTA pair keeps one ROW tile (256 rows x dpad, 128 KB per CTA) resident in shared
// memory and streams the QUERY tiles past it through the TMA ring.  The query matrix is a few MB
// and stays hot in L2, every row of the shard is fetched from HBM exactly ONCE per search, and the
// row tiles are simply split evenly over the pairs (no lockstep needed).  The accumulator is still
// [queries x rows], so the epilogue is unchanged except that a thread's query changes with every
// unit: its list / count live in per-(pair, set, query) arrays, its threshold is the per-query
// threshold shared by all CTAs, and the lists are folded directly by the merge kernel (no flush).
// ===================================================================================
struct XresParams {
    int64_t n_rows;
    int     nq, k, C, kblocks, stages, tq;
    int64_t nt;              // row tiles of this launch
    int64_t tile0;           // first row tile of this launch
    int     tn;              // rows per tile (256, 192 or 128)
    int     groups;          // CTA pairs
    int     nq_pad;          // tq * 256
    uint64_t* lists;         // [groups][2 sets][nq_pad / 32][C][32] raw candidate lists, interleaved per warp
    int*      counts;        // [groups][2 sets][nq_pad]
    uint32_t* tau_g;         // [nq_pad] shared per-query threshold (order-preserving encoding)
    uint64_t  row_policy;
    int       prefetch;        // pull the next row tile into L2 halfway through the current one
    int       skip_epilogue;   // debug/perf probe: drain nothing (results are garbage)
};

// TN = rows per tile: 256 for dpad <= 512, 224 (or 192) for dpad <= 768, 128 (or 160) for dpad <= 1024.
template <int E, int TN>
__global__ void __launch_bounds__(kMmaThreads, 1)
search_mma_xres_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_x,
                       const XresParams p) {
    constexpr int CG = 2;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cta_rank = cluster_ctarank();
    const int group = blockIdx.x / CG;

    constexpr uint32_t stage_bytes = kTileQ * 128;               // one query k-block per CTA: 16 KB
    constexpr uint32_t x_block = (TN / CG) * 128;                 // one k-block of this CTA's half of the row tile
    const uint32_t x_bytes = p.kblocks * x_block;
    const uint32_t smem_x = smem_base;
    const uint32_t smem_s = smem_x + x_bytes;
    const uint32_t bars = smem_s + p.stages * stage_bytes;
    auto full_bar  = [&](int s) { return bars + 8u * s; };
    auto empty_bar = [&](int s) { return bars + 8u * (16 + s); };
    const uint32_t x_full = bars + 8u * 32, x_empty = bars + 8u * 33;
    auto tfull_bar  = [&](int a) { return bars + 8u * (34 + a); };
    auto tempty_bar = [&](int a) { return bars + 8u * (36 + a); };
    const uint32_t tmem_slot = bars + 8u * 40;

    const int64_t j0 = p.nt * group / p.groups, j1 = p.nt * (group + 1) / p.groups;   // owned row tiles

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        mbar_init(x_full, 1); mbar_init(x_empty, 1);
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4 * CG); }
        fence_barrier_init();
    }
    if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmap_q); tma_prefetch_desc(&tmap_x); }
    if (warp == 2) tmem_alloc<CG>(tmem_slot, 512);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    if (warp == 0 && lane == 0) {
        // ============================ TMA producer ============================
        int stage = 0; uint32_t phase = 0; int nload = 0;
        for (int64_t j = j0; j < j1; ++j) {
            bool pending = true; int issued = 0;
            auto load_x = [&]() {
                if (nload > 0) mbar_wait(x_empty, (nload - 1) & 1);  // MMAs finished with the old row tile
                if (cta_rank == 0) mbar_expect_tx(x_full, x_bytes * CG);
                for (int kb = 0; kb < p.kblocks; ++kb)
                    tma_load_2d<CG>(smem_x + kb * x_block, &tmap_x, x_full, kb * kKBlock,
                                    static_cast<int>((p.tile0 + j) * TN) + static_cast<int>(cta_rank) * (TN / CG), p.row_policy);
                ++nload;
                pending = false;
            };
            if (nload == 0) load_x();
            for (int t = 0; t < p.tq; ++t) {
                if (p.prefetch && t == p.tq / 2 && j + 1 < j1) {
                    // pull the next row tile into L2 while this one is being used
                    for (int kb = 0; kb < p.kblocks; ++kb)
                        asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];"
                                     ::"l"(reinterpret_cast<uint64_t>(&tmap_x)), "r"(kb * kKBlock),
                                       "r"(static_cast<int>((p.tile0 + j + 1) * TN) + static_cast<int>(cta_rank) * (TN / CG))
                                     : "memory");
                }
                for (int kb = 0; kb < p.kblocks; ++kb) {
                    if (pending && issued >= p.stages) load_x();     // ring refilled first, then the row tile
                    mbar_wait(empty_bar(stage), phase ^ 1);
                    if (cta_rank == 0) mbar_expect_tx(full_bar(stage), stage_bytes * CG);
                    tma_load_2d<CG>(smem_s + stage * stage_bytes, &tmap_q, full_bar(stage), kb * kKBlock,
                                    t * (kTileQ * CG) + static_cast<int>(cta_rank) * kTileQ, kL2EvictLast);
                    ++issued;
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
            }
            if (pending) load_x();
        }
        // This thread consumed every x_empty completion but the last, in order: waiting for the last
        // one here is unambiguous and keeps the CTA alive until no asynchronous arrive is in flight.
        if (nload > 0) mbar_wait(x_empty, (nload - 1) & 1);
    } else if (warp == 1 && lane == 0) {
        // ============================ MMA issuer (leader CTA) =================
        constexpr uint32_t idesc = make_idesc(kTileQ * CG, TN);
        int stage = 0; uint32_t phase = 0; int nload = 0; int64_t n = 0;
        for (int64_t j = j0; j < j1; ++j) {
            if (cta_rank == 0) mbar_wait(x_full, nload & 1);
            ++nload;
            if (cta_rank == 0) {
                for (int t = 0; t < p.tq; ++t, ++n) {
                    const int acc = static_cast<int>(n & 1);
                    const uint32_t acc_phase = static_cast<uint32_t>((n >> 1) & 1);
                    mbar_wait(tempty_bar(acc), acc_phase ^ 1);
                    tc_fence_after();
                    const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(acc * TN);
                    for (int kb = 0; kb < p.kblocks; ++kb) {
                        mbar_wait(full_bar(stage), phase);
                        tc_fence_after();
                        const uint32_t a0 = smem_s + stage * stage_bytes;       // A: streamed query k-block
                        const uint32_t b0 = smem_x + kb * x_block;               // B: resident row-tile k-block
#pragma unroll
                        for (int k4 = 0; k4 < kKBlock / 16; ++k4)
                            umma_f16<CG>(tmem_d, make_smem_desc(a0 + k4 * 32), make_smem_desc(b0 + k4 * 32), idesc,
                                         (kb | k4) ? 1u : 0u);
                        umma_commit<CG>(empty_bar(stage));
                        if (++stage == p.stages) { stage = 0; phase ^= 1; }
                    }
                    umma_commit<CG>(tfull_bar(acc));
                }
                umma_commit<CG>(x_empty);                           // row tile released when its MMAs retire
            }
        }
    } else if (warp >= 4) {
        // ============================ epilogue: fused top-k ====================
        const int set = (warp - 4) >> 2;
        const int quarter = warp & 3;
        const int r = quarter * 32 + lane;
        const float POS_INF = __int_as_float(0x7f800000);
        const int64_t set_base = (static_cast<int64_t>(group) * 2 + set) * p.nq_pad;
        int cnt = 0; float tau = 0.f; int64_t q_global = 0; bool q_ok = false;
        uint64_t* my_list = nullptr;
        // state of this set's NEXT unit, prefetched while the current one is processed
        int64_t pf_n = -1; int pf_cnt = 0; uint32_t pf_tau = 0;
        auto q_of = [&](int t) { return static_cast<int64_t>(t) * (kTileQ * CG) + cta_rank * kTileQ + r; };

        // make room for two more chunks (<= 64 entries): all 32 lists of the warp are pruned together
        auto make_room = [&]() {
            if (!__any_sync(0xffffffffu, cnt > p.C - 64)) return;
            const float tau_before = tau;
            unsigned bad = warp_prune_lists(my_list, cnt, tau, p.k);
            bad |= __ballot_sync(0xffffffffu, cnt > p.C - 64);      // no pivot / no progress (ties): exact compaction
            while (bad) {
                const int l = __ffs(bad) - 1; bad &= bad - 1;
                const int c_l = __shfl_sync(0xffffffffu, cnt, l);
                __syncwarp();
                const float t_l = warp_compact_raw<E>(my_list - lane + l, c_l, p.k, p.C, lane, kListStride);
                if (lane == l) { cnt = min(cnt, p.k); tau = fmaxf(tau, t_l); }
            }
            if (q_ok && tau > tau_before) atomicMax(p.tau_g + q_global, f2ord(tau));
        };
        auto process_chunk = [&](uint32_t (&v)[32], int c, int64_t row0, int nvalid) {
            if (IVR_SKIP_EPI(p) == 2) return;                        // perf probe: tcgen05.ld traffic only
            filter_chunk(v, tau, cnt, my_list, static_cast<uint32_t>(row0) + c * 32, c * 32, nvalid, TN);
        };

        const int64_t n_units = (j1 - j0) * p.tq;
        // (j, t) of unit n advance by two units per iteration without divisions
        int64_t j = j0 + set / p.tq;
        int t = set % p.tq;
        const int step_j = 2 / p.tq, step_t = 2 % p.tq;
        for (int64_t n = set; n < n_units; n += 2) {
            q_global = q_of(t);
            q_ok = q_global < p.nq;
            const int64_t idx = set_base + q_global;
            if (pf_n == n) { cnt = pf_cnt; tau = ord2f(pf_tau); }
            else { cnt = p.counts[idx]; tau = ord2f(__ldcg(p.tau_g + q_global)); }
            if (!q_ok) tau = POS_INF;                               // padded queries admit nothing
            my_list = p.lists + (idx - lane) * p.C + lane;       // interleaved: entry i at my_list[i * 32]
            int t2 = t + step_t; int64_t j2 = j + step_j;
            if (t2 >= p.tq) { t2 -= p.tq; ++j2; }
            if (n + 2 < n_units) {                                  // prefetch the state of unit n + 2
                const int64_t q2 = q_of(t2);
                pf_n = n + 2; pf_cnt = p.counts[set_base + q2]; pf_tau = __ldcg(p.tau_g + q2);
            }
            const int64_t row0 = (p.tile0 + j) * TN;
            const int nvalid = static_cast<int>(min(static_cast<int64_t>(TN), p.n_rows - row0));
            mbar_wait(tfull_bar(set), static_cast<uint32_t>((n >> 1) & 1));
            tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) +
                                   static_cast<uint32_t>(set * TN);
            uint32_t va[32], vb[32];
            if (IVR_SKIP_EPI(p) != 1) tmem_ld_32x32(taddr, va);
#pragma unroll 1
            for (int c = 0; c < (IVR_SKIP_EPI(p) == 1 ? 0 : TN / 32); c += 2) {
                make_room();
                tmem_wait_ld(va);
                const bool pair = (TN / 32) % 2 == 0 || c + 1 < TN / 32;    // TN = 224: seven chunks, the last one alone
                if (pair) tmem_ld_32x32(taddr + (c + 1) * 32, vb);
                process_chunk(va, c, row0, nvalid);
                if (pair) {
                    tmem_wait_ld(vb);
                    if (c + 2 < TN / 32) tmem_ld_32x32(taddr + (c + 2) * 32, va);
                    process_chunk(vb, c + 1, row0, nvalid);
                }
            }
            p.counts[idx] = cnt;
            // the same query comes back when the next row tile is swept; when tq is odd the prefetched
            // count of unit n + 2 could be this very slot only if tq == 2 -- excluded: tq == 2 => n + 2 has the same t
            if (pf_n == n + 2 && t2 == t) pf_cnt = cnt;
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(tempty_bar(set), 0);
            t = t2; j = j2;
        }
    }

    // ------------------------------------------------------------------ teardown ----
    tc_fence_before();
    cluster_sync_all();
    if (warp == 2) tmem_dealloc<CG>(tmem_base, 512);
}

// fp32 [nq, dim] -> fp16 [nq_pad, dpad] (zero padded), one warp per query.  Each query is scaled by
// a power of two so that its largest component lies in [0.5, 1): exact, keeps fp16 in range for
// any query norm, and is undone on the final scores (scale[q]).  The exponent is clamped to [-127, 127] so that
// both 2^e and 2^-e are finite fp32: below 2^-128 the largest component lands under 0.5, from 2^128 * 0.5 up in
// [1, 2); a zero or non-finite maximum keeps e = 0.
__global__ void queries_to_f16_kernel(const float* __restrict__ q, __half* __restrict__ out,
                                      float* __restrict__ scale, uint32_t* __restrict__ tau_g,
                                      int64_t nq, int64_t nq_pad, int dim, int dpad) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
    if (r >= nq_pad) return;
    float mx = 0.f;
    if (r < nq)
        for (int c = lane; c < dim; c += 32) mx = fmaxf(mx, fabsf(q[r * dim + c]));
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    int e = 0;
    if (mx > 0.f && isfinite(mx)) {
        frexpf(mx, &e);                                            // mx = m * 2^e, m in [0.5, 1)
        e = min(max(e, -127), 127);
    }
    const float down = ldexpf(1.0f, -e);
    for (int c = lane; c < dpad; c += 32)
        out[r * dpad + c] = __float2half_rn((r < nq && c < dim) ? q[r * dim + c] * down : 0.f);
    if (lane == 0) {
        scale[r] = ldexpf(1.0f, e);
        tau_g[r] = f2ord(__int_as_float(0xff800000));             // shared threshold starts at -inf
    }
}


// Between launches: every query's shared threshold starts the next launch at the EXACT k-th
// best score of the rows searched by the previous one (a valid lower bound of the final k-th best), in the kernel's
// scaled score domain (keys hold unscaled-by-q_scale scores, i.e. already that domain).
__global__ void seed_tau_kernel(const uint64_t* __restrict__ keys, const int* __restrict__ counts,
                                uint32_t* __restrict__ tau_g, int64_t nq, int k) {
    const int64_t q = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (q >= nq) return;
    if (counts[q] >= k) atomicMax(tau_g + q, f2ord(key_score(keys[q * k + k - 1])));
}

// ------------------------------------------------------------------ host side ----
int launch_queries_to_f16(const float* q, __half* out, float* scale, uint32_t* tau_g, int64_t nq, int64_t nq_pad,
                          int dim, int dpad, cudaStream_t st) {
    const int64_t threads = nq_pad * 32;
    queries_to_f16_kernel<<<static_cast<unsigned>((threads + 255) / 256), 256, 0, st>>>(q, out, scale, tau_g, nq, nq_pad, dim, dpad);
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

int row_tmap(ivr_index* idx, int box_rows, const CUtensorMap** tmx) {
    if (idx->tmap_rows_base != idx->rows || idx->tmap_rows_n != idx->ntotal || idx->tmap_rows_box != box_rows) {
        IVR_TRY(make_tmap(reinterpret_cast<CUtensorMap*>(idx->tmap_rows), idx->rows, idx->ntotal, idx->dpad, box_rows));
        idx->tmap_rows_base = idx->rows; idx->tmap_rows_n = idx->ntotal; idx->tmap_rows_box = box_rows;
    }
    *tmx = reinterpret_cast<const CUtensorMap*>(idx->tmap_rows);
    return IVR_OK;
}

int prepare_queries(ivr_index* idx, bool timed, const float* q_dev, int64_t nq, int64_t nq_pad, __half* q_h,
                    float* q_scale, uint32_t* tau_g, int box_rows, CUtensorMap* tmq, cudaStream_t st,
                    void* zero, size_t zero_bytes) {
    timing_mark(idx, timed, kPrepBegin, st);
    IVR_TRY(launch_queries_to_f16(q_dev, q_h, q_scale, tau_g, nq, nq_pad, idx->dim, idx->dpad, st));
    if (zero_bytes) IVR_CUDA(cudaMemsetAsync(zero, 0, zero_bytes, st));
    idx->launches[2]++;
    timing_mark(idx, timed, kPrepEnd, st);
    return make_tmap(tmq, q_h, nq_pad, idx->dpad, box_rows);
}

int begin_launches(LaunchSeq* seq, int64_t nq_pad, int max_lists, size_t own_bytes) {
    const int64_t nq = seq->nq;
    const int k = seq->k;
    Carve carve;
    const size_t o_q  = carve(static_cast<size_t>(nq_pad) * seq->idx->dpad * 2);
    const size_t o_sc = carve(static_cast<size_t>(nq_pad) * 4);
    const size_t o_tg = carve(static_cast<size_t>(nq_pad) * 4);
    const size_t o_pk = carve(static_cast<size_t>(seq->n) * nq * k * 8);
    const size_t o_pc = carve(static_cast<size_t>(seq->n) * nq * 4);
    const size_t o_t  = carve(merge_tmp_entries(max_lists, nq, k) * 8);
    const size_t o_tc = carve((static_cast<size_t>(max_lists) * nq + 64) * 4);
    const size_t o_own = carve(own_bytes);
    IVR_TRY(ensure_ws(seq->idx, carve.size));
    char* ws = static_cast<char*>(seq->idx->ws);
    seq->q_h = reinterpret_cast<__half*>(ws + o_q);
    seq->q_scale = reinterpret_cast<float*>(ws + o_sc);
    seq->tau_g = reinterpret_cast<uint32_t*>(ws + o_tg);
    seq->keys = reinterpret_cast<uint64_t*>(ws + o_pk);
    seq->counts = reinterpret_cast<int*>(ws + o_pc);
    seq->tmp_e = reinterpret_cast<uint64_t*>(ws + o_t);
    seq->tmp_c = reinterpret_cast<int*>(ws + o_tc);
    seq->own = ws + o_own;
    return IVR_OK;
}

int fold_launch(LaunchSeq& s, int ph, const MergeIn& lists) {
    if (s.n == 1) {
        timing_mark(s.idx, s.timed, kScoreEnd, s.st); timing_mark(s.idx, s.timed, kMergeBegin, s.st);
        return merge_lists_final(lists, s.nq, s.k, s.D, s.I, s.id_offset, s.tmp_e, s.tmp_c, s.st, &s.idx->launches[1],
                                 s.q_scale);
    }
    uint64_t* keys = s.keys + static_cast<size_t>(ph) * s.nq * s.k;
    int* counts = s.counts + static_cast<size_t>(ph) * s.nq;
    IVR_TRY(merge_lists_keys(lists, s.nq, s.k, keys, counts, s.tmp_e, s.tmp_c, s.st, &s.idx->launches[1]));
    if (ph + 1 < s.n) {
        // the k-th best of this launch: tau_g already holds the earlier launches' (atomicMax: the seed can only rise)
        seed_tau_kernel<<<static_cast<unsigned>((s.nq + 255) / 256), 256, 0, s.st>>>(keys, counts, s.tau_g, s.nq, s.k);
        IVR_CUDA(cudaGetLastError());
        s.idx->launches[1]++;
    }
    return IVR_OK;
}

int finish_launches(LaunchSeq& s) {
    if (s.n > 1) {
        timing_mark(s.idx, s.timed, kScoreEnd, s.st); timing_mark(s.idx, s.timed, kMergeBegin, s.st);
        MergeIn in{};
        in.entries = s.keys; in.counts = s.counts;
        in.list_stride = s.nq * s.k; in.q_stride = s.k; in.cnt_list_stride = s.nq; in.cnt_q_stride = 1;
        in.n_lists = s.n; in.fixed_count = 0; in.raw = 0;
        IVR_TRY(merge_lists_final(in, s.nq, s.k, s.D, s.I, s.id_offset, s.tmp_e, s.tmp_c, s.st, &s.idx->launches[1],
                                  s.q_scale));
    }
    timing_mark(s.idx, s.timed, kMergeEnd, s.st);
    if (s.timed) s.idx->ev_valid[0] = s.idx->ev_valid[1] = s.idx->ev_valid[2] = true;
    return IVR_OK;
}

// IVR_MMA_CTA_GROUP=1 / 2 forces single CTAs / CTA pairs (cta_group::2) for the query-tile-resident kernel;
// read per call so tests can flip it.
// Unset / 0: CTA pairs unless single CTAs (128-query tiles) multiply at least 25 % less padding -- measured on the
// query-tile-resident kernel, 10 M rows: 128 queries 2.01 ms (single CTAs) vs 2.38 ms (pairs), 384: 4.36 vs 4.79,
// 192 / 256: 2.87 / 3.14 vs 2.52 / 2.71; 100 M x 128 queries: 19.0 vs 25.1 ms.
static int cta_group_mode(int64_t nq) {
    const int e = env_int("IVR_MMA_CTA_GROUP", 0);
    if (e == 1 || e == 2) return e;
    const int64_t pad1 = (nq + kTileQ - 1) / kTileQ * kTileQ, pad2 = (nq + 2 * kTileQ - 1) / (2 * kTileQ) * (2 * kTileQ);
    return pad1 * 4 <= pad2 * 3 ? 1 : 2;
}

bool mma_supported(const ivr_index* idx, int64_t nq, int k) {
    (void)nq;
    return idx->dpad <= 2 * kMaxKBlocks * kKBlock && k <= IVR_MAX_K;     // up to 1024 dims
}

// ---- launch plans ---------------------------------------------------------------------
// A plan describes one scoring launch over the row tiles [tile0, tile0 + nt): kernel parameters,
// the scratch it needs, and how the merge kernel reads the candidate lists it leaves behind.
struct Plan {
    bool      xres = false;
    int       cg = 2, grid = 0, E = 8;
    size_t    smem = 0;
    MmaParams q{};            // query-tile-resident
    XresParams x{};           // row-tile-resident
    size_t    list_bytes = 0, aux_bytes = 0;    // lists; state / counts / slot buffers
    int       n_lists = 0;
};

static int plan_qres(const ivr_index* idx, int cg, int64_t nq, int k, int64_t tile0, int64_t nt, Plan* pl) {
    const int C = 2 * kcap_for(k);
    const int mq = kTileQ * cg;
    MmaParams& p = pl->q;
    p = MmaParams{};
    p.n_rows = idx->ntotal; p.nq = static_cast<int>(nq); p.k = k; p.C = C;
    p.kblocks = idx->dpad / kKBlock;
    p.tq = static_cast<int>((nq + mq - 1) / mq);
    p.nt = nt; p.tile0 = tile0;
    p.nq_pad = p.tq * mq;
    int grid = idx->sm_count / cg * cg;
    p.groups = grid / cg;                                          // caller guarantees tq <= groups
    p.c = p.groups / p.tq;
    p.g_grid = p.c * p.tq;
    p.ntg = (p.g_grid == p.groups) ? p.nt : (p.nt * p.g_grid + p.groups / 2) / p.groups;
    if (p.nt - p.ntg > 0 && static_cast<int64_t>(p.tq) * (p.nt - p.ntg) < p.groups - p.g_grid) p.ntg = p.nt;
    p.stagger = std::max(0, env_int("IVR_MMA_STAGGER", 1));
#ifdef IVR_PROBES
    p.skip_epilogue = env_int("IVR_MMA_DEBUG_SKIP_EPILOGUE", 0);
#endif
    {
        const int pol = env_int("IVR_MMA_ROW_POLICY", 0);          // 0 normal, 1 evict-first, 2 evict-last
        p.row_policy = pol == 1 ? kL2EvictFirst : (pol == 2 ? kL2EvictLast : kL2EvictNormal);
    }
    const int stage_bytes = (kTileN / cg) * 128;
    const int q_bytes = p.kblocks * kQBlockBytes;
    p.stages = std::min(12, (kSmemBudget - 1024 - kBarrierBytes - q_bytes) / stage_bytes);
    if (p.stages < 2) { set_error("search_mma: dim %d leaves no room for the row-tile ring", idx->dim); return IVR_EUNSUPPORTED; }
    pl->smem = 1024 + q_bytes + static_cast<size_t>(p.stages) * stage_bytes + kBarrierBytes;
    const int Gl = p.groups - p.g_grid;
    const int64_t ntl = p.nt - p.ntg, Ul = static_cast<int64_t>(p.tq) * ntl;
    int left_per_tile = 0;
    p.segs_max = 1;
    if (Gl > 0 && Ul > 0) {
        auto gl_of = [&](int64_t u) { return static_cast<int>(((u + 1) * Gl - 1) / Ul); };
        for (int t = 0; t < p.tq; ++t)
            left_per_tile = std::max(left_per_tile, gl_of(static_cast<int64_t>(t) * ntl + ntl - 1) -
                                                    gl_of(static_cast<int64_t>(t) * ntl) + 1);
        for (int g = 0; g < Gl; ++g) {
            const int64_t ub = Ul * g / Gl, ue = Ul * (g + 1) / Gl;
            if (ue > ub) p.segs_max = std::max(p.segs_max, static_cast<int>((ue - 1) / ntl - ub / ntl) + 1);
        }
    }
    pl->xres = false; pl->cg = cg; pl->grid = grid; pl->E = (C == 256) ? 8 : 0;
    pl->n_lists = 2 * (p.c + left_per_tile);                       // output slots per query
    pl->list_bytes = static_cast<size_t>(pl->n_lists) * p.nq_pad * C * 8;
    pl->aux_bytes = static_cast<size_t>(grid) * p.segs_max * 2 * kTileQ * sizeof(int2) + 256 +
                    static_cast<size_t>(pl->n_lists) * p.nq_pad * 4 + 256;
    return IVR_OK;
}

// rows per resident tile: the largest UMMA N whose half tile (N/2 rows x dpad fp16 per CTA) leaves room for the
// query ring -- 256 up to 512 dims, 192 up to 768 (N = 128 costs 1.5x the shared-memory operand traffic per
// FLOP: measured 926 TFLOP/s pipeline-only at 768 dims), 128 up to 1024
static int xres_tile_rows(const ivr_index* idx) {
    if (idx->dpad <= 512) return 256;
    // 768 dims: N = 224 (168 KB resident per CTA, 3-stage query ring) beats N = 192 (144 KB, 5 stages): 10 M x 768 x
    // 4096 queries 56.7 -> 51.8 ms, x 16384: 219 -> 200 ms (the wider tile reads less shared memory per FLOP)
    if (idx->dpad <= 768) { const int t = env_int("IVR_XRES_TN_768", 224); return (t == 192 || t == 256) ? t : 224; }
    // 1024 dims: N = 160 (160 KB resident, 4 stages) beats N = 128 (128 KB, 6 stages): 5 M x 1024 x 4096 queries 47.8 -> 42.9 ms
    { const int t = env_int("IVR_XRES_TN_1024", 160); return (t == 128 || t == 192) ? t : 160; }
}

static int plan_xres(const ivr_index* idx, int64_t nq, int k, int64_t tile0, int64_t nt, Plan* pl) {
    constexpr int cg = 2;
    const int C = 2 * kcap_for(k);
    const int mq = kTileQ * cg;
    XresParams& p = pl->x;
    p = XresParams{};
    p.n_rows = idx->ntotal; p.nq = static_cast<int>(nq); p.k = k; p.C = C;
    p.kblocks = idx->dpad / kKBlock;
    p.tq = static_cast<int>((nq + mq - 1) / mq);
    p.nt = nt; p.tile0 = tile0;
    p.nq_pad = p.tq * mq;
    int grid = idx->sm_count / cg * cg;
    p.groups = grid / cg;
    if (p.nt < p.groups) { p.groups = static_cast<int>(std::max<int64_t>(p.nt, 1)); grid = p.groups * cg; }
#ifdef IVR_PROBES
    p.skip_epilogue = env_int("IVR_MMA_DEBUG_SKIP_EPILOGUE", 0);
#endif
    {
        const int pol = env_int("IVR_MMA_ROW_POLICY", 1);          // rows are read once: evict-first by default
        p.row_policy = pol == 1 ? kL2EvictFirst : (pol == 2 ? kL2EvictLast : kL2EvictNormal);
    }
    p.prefetch = env_int("IVR_XRES_PREFETCH", 1);
    p.tn = xres_tile_rows(idx);
    const int stage_bytes = kTileQ * 128;
    const int x_bytes = p.kblocks * (p.tn / cg) * 128;
    p.stages = std::min(12, (kSmemBudget - 1024 - kBarrierBytes - x_bytes) / stage_bytes);
    if (p.stages < 2) { set_error("search_mma: dim %d leaves no room for the query ring", idx->dim); return IVR_EUNSUPPORTED; }
    pl->smem = 1024 + x_bytes + static_cast<size_t>(p.stages) * stage_bytes + kBarrierBytes;
    pl->xres = true; pl->cg = cg; pl->grid = grid; pl->E = (C == 256) ? 8 : 0;
    pl->n_lists = p.groups * 2;
    pl->list_bytes = static_cast<size_t>(pl->n_lists) * p.nq_pad * C * 8;
    pl->aux_bytes = static_cast<size_t>(pl->n_lists) * p.nq_pad * 4 + 256;
    return IVR_OK;
}

template <typename Kern, typename Params>
static int launch_cluster(Kern kern, const CUtensorMap& tq, const CUtensorMap& tx, const Params& p, int grid, int cg,
                          size_t smem, cudaStream_t st) {
    IVR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(kMmaThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cg; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    IVR_CUDA(cudaLaunchKernelEx(&cfg, kern, tq, tx, p));
    return IVR_OK;
}

// The instantiations run_plan picks from, in the order they are instantiated (the order of the kernels in the
// module, which can change their register allocation): search_mma_xres_kernel<E, TN> by
// [(256 - TN) / 32][E == 0] for the tile heights of xres_tile_rows(), search_mma_kernel<CG, E> by [2 - CG][E == 0].
using XresKernel = void (*)(const CUtensorMap, const CUtensorMap, const XresParams);
using QresKernel = void (*)(const CUtensorMap, const CUtensorMap, const MmaParams);
static const XresKernel kXresKernels[5][2] = {
    {search_mma_xres_kernel<8, 256>, search_mma_xres_kernel<0, 256>},
    {search_mma_xres_kernel<8, 224>, search_mma_xres_kernel<0, 224>},
    {search_mma_xres_kernel<8, 192>, search_mma_xres_kernel<0, 192>},
    {search_mma_xres_kernel<8, 160>, search_mma_xres_kernel<0, 160>},
    {search_mma_xres_kernel<8, 128>, search_mma_xres_kernel<0, 128>}};
static const QresKernel kQresKernels[2][2] = {{search_mma_kernel<2, 8>, search_mma_kernel<2, 0>},
                                              {search_mma_kernel<1, 8>, search_mma_kernel<1, 0>}};

// Runs one planned launch with its scratch at `lists` / `aux`; fills `in` for the merge kernel.
static int run_plan(Plan& pl, const CUtensorMap& tmq, const CUtensorMap& tmx, uint32_t* tau_g, char* lists, char* aux,
                    cudaStream_t st, MergeIn* in) {
    const int e0 = pl.E != 8;
    int64_t nq_pad;
    int C;
    int* counts;
    if (pl.xres) {
        XresParams& p = pl.x;
        p.tau_g = tau_g;
        p.lists = reinterpret_cast<uint64_t*>(lists);
        p.counts = counts = reinterpret_cast<int*>(aux);
        IVR_CUDA(cudaMemsetAsync(p.counts, 0, static_cast<size_t>(pl.n_lists) * p.nq_pad * 4, st));
        IVR_TRY(launch_cluster(kXresKernels[(256 - p.tn) / 32][e0], tmq, tmx, p, pl.grid, 2, pl.smem, st));
        nq_pad = p.nq_pad; C = p.C;
    } else {
        MmaParams& p = pl.q;
        p.tau_g = tau_g;
        p.lists = reinterpret_cast<uint64_t*>(lists);
        Carve carve;
        p.state = reinterpret_cast<int2*>(aux + carve(static_cast<size_t>(pl.grid) * p.segs_max * 2 * kTileQ * sizeof(int2)));
        p.counts = counts = reinterpret_cast<int*>(aux + carve(static_cast<size_t>(pl.n_lists) * p.nq_pad * 4));
        IVR_CUDA(cudaMemsetAsync(p.counts, 0, static_cast<size_t>(pl.n_lists) * p.nq_pad * 4, st));
        IVR_TRY(launch_cluster(kQresKernels[2 - pl.cg][e0], tmq, tmx, p, pl.grid, pl.cg, pl.smem, st));
        nq_pad = p.nq_pad; C = p.C;
    }
    *in = MergeIn{};
    in->entries = reinterpret_cast<const uint64_t*>(lists); in->counts = counts;
    in->list_stride = nq_pad * C; in->q_stride = C;
    in->cnt_list_stride = nq_pad; in->cnt_q_stride = 1;
    in->n_lists = pl.n_lists; in->fixed_count = 0; in->raw = 1; in->interleave = 1;
    return IVR_OK;
}

// One query batch.  The shard is searched in several launches of growing size: the exact k-th best score
// per query of one launch seeds the shared admission thresholds of the next -- the fused top-k epilogue
// admits ~k * ratio candidates per launch instead of re-learning its thresholds in every list
// (measured: 22k-45k admissions per query in a single launch).
static int search_mma_batch(ivr_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev,
                            int64_t id_offset, cudaStream_t st, int cg, bool xres, bool first_batch) {
    const int mq = kTileQ * (xres ? 2 : cg);
    const int tq = static_cast<int>((nq + mq - 1) / mq);
    const int64_t nq_pad = static_cast<int64_t>(tq) * mq;
    const int tile_rows = xres ? xres_tile_rows(idx) : kTileN;     // both phases use the same tile size
    const int64_t nt = (idx->ntotal + tile_rows - 1) / tile_rows;
    // Launch boundaries (in row tiles).  The first launch covers a small prefix (IVR_MMA_PHASE0_ROWS, 2 k rows), every
    // further one IVR_MMA_PHASE_RATIO times the rows seen so far, the last one the rest: a launch then admits
    // ~k * ratio candidates per query instead of re-learning its thresholds in every list.  If the last launch would
    // still be more than `ratio` times the rows seen before it, one more boundary goes to the geometric mean (1 M rows
    // at ratio 16: 2 k, 32 k, REST = 30 x was 4.5 ms for 4096 queries against 3.6 ms with an even split).
    // First launch: 8 k rows until the merges between launches became cheap (topk_merge.cu, flattened select); with
    // them 2 k rows win on small shards -- 100 k x 1000 queries 0.44 -> 0.32 ms, 1 M x 256 0.49 -> 0.42 ms, 1 M x 1024
    // 1.16 -> 1.03-1.12 ms -- and are neutral from 10 M rows up (profiles/r2_phase_schedule_after_merge.txt).
    constexpr int kMaxPhases = 7;
    int64_t bounds[kMaxPhases + 1] = {0};
    int n_phases = 0;
    if (env_int("IVR_MMA_TWO_PHASE", 1)) {
        // the row-tile-resident kernel spreads a query over 148 lists that never fill up during one launch, so
        // its thresholds only improve at launch boundaries: it gets more of them (measured, 10 M x 4096 queries:
        // 34.0 ms at ratio 8 vs 35.5 ms at 16; the query-tile-resident kernel prefers 16: 8.4 vs 8.9 ms at 1024 queries)
        const int64_t ratio = std::max(2, env_int("IVR_MMA_PHASE_RATIO", xres ? 8 : 16));
        int64_t b = std::max<int64_t>(1, env_int("IVR_MMA_PHASE0_ROWS", 2048) / tile_rows);
        while (n_phases < kMaxPhases - 2 && b * 2 <= nt) {         // a boundary must leave at least as much for later
            bounds[++n_phases] = b;
            b *= ratio;
        }
        if (n_phases > 0 && nt > bounds[n_phases] * ratio) {
            const int64_t g = static_cast<int64_t>(std::sqrt(static_cast<double>(bounds[n_phases]) * static_cast<double>(nt)));
            if (g > bounds[n_phases] && g < nt) bounds[++n_phases] = g;
        }
    }
    bounds[++n_phases] = nt;
    Plan plan[kMaxPhases];
    for (int ph = 0; ph < n_phases; ++ph) {
        const int64_t t0 = bounds[ph], n = bounds[ph + 1] - bounds[ph];
        // the early launches have to learn their thresholds from scratch: the query-tile-resident kernel
        // (few, long candidate streams per query) does that better, so it runs every launch but the last
        // whenever the layouts agree (CTA pairs, one query tile per pair available, 256-row tiles)
        // -- and the launch is short (<= 3 M rows: beyond that re-reading the rows per query tile costs more)
        const bool early_qres = xres && ph + 1 < n_phases && cg == 2 && tq <= idx->sm_count / 2 && tile_rows == kTileN &&
                                n * tile_rows <= static_cast<int64_t>(env_int("IVR_MMA_EARLY_QRES_MAX_KROWS", 3000)) * 1000;
        IVR_TRY((xres && !early_qres) ? plan_xres(idx, nq, k, t0, n, &plan[ph]) : plan_qres(idx, cg, nq, k, t0, n, &plan[ph]));
    }
    size_t list_bytes = 0, aux_bytes = 0; int max_lists = 2;
    for (int ph = 0; ph < n_phases; ++ph) {
        list_bytes = std::max(list_bytes, plan[ph].list_bytes);
        aux_bytes = std::max(aux_bytes, plan[ph].aux_bytes);
        max_lists = std::max(max_lists, plan[ph].n_lists);
    }
    Carve own;
    const size_t o_l = own(list_bytes), o_a = own(aux_bytes);
    LaunchSeq seq{idx, st, idx->timing && first_batch, nq, k, n_phases, D_dev, I_dev, id_offset};
    IVR_TRY(begin_launches(&seq, nq_pad, max_lists, own.size));

    CUtensorMap tmq;
    const CUtensorMap* tmx;
    const int box_rows = tile_rows / (xres ? 2 : cg);
    IVR_TRY(prepare_queries(idx, seq.timed, q_dev, nq, nq_pad, seq.q_h, seq.q_scale, seq.tau_g, kTileQ, &tmq, st));
    IVR_TRY(row_tmap(idx, box_rows, &tmx));

    timing_mark(idx, seq.timed, kScoreBegin, st);
    for (int ph = 0; ph < n_phases; ++ph) {
        MergeIn in;
        IVR_TRY(run_plan(plan[ph], tmq, *tmx, seq.tau_g, seq.own + o_l, seq.own + o_a, st, &in));
        idx->launches[0]++;
        IVR_TRY(fold_launch(seq, ph, in));
    }
    return finish_launches(seq);
}

int search_mma(ivr_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev,
               int64_t id_offset, cudaStream_t st) {
    // Mode selection: IVR_MMA_MODE = 0 auto, 1 query-tile-resident, 2 row-tile-resident, 3 small-batch.
    // Auto: the small-batch (row-streaming) kernel up to IVR_MMA_SMALL_MAX_NQ queries where its shape fits;
    // the row-tile-resident kernel (cta_group::2) from 4 query tiles (> 768 queries) up on large shards.
    const int mode = env_int("IVR_MMA_MODE", 0);
    const int cg = cta_group_mode(nq);
    // measured (10 M rows): 512 dims -- 64 queries 2.0 ms small-batch vs 2.1 ms batched, 80: 2.5 vs 2.2, 128: 3.7 vs 2.3
    // (the resident queries squeeze the row ring); 768 dims -- 64..80 queries 2.4-2.6 ms vs 5.7-6.2 ms
    // Round 2, after the merges between launches became cheap, the batched kernel (single CTAs, M = 128) took over
    // 17..64 queries on large shards: 10 M rows -- 24 / 32 / 48 / 64 queries 1.72 / 1.73 / 1.76 / 1.76 ms against
    // 1.80 / 1.78 / 2.12 / 2.19 ms on the small-batch kernel; 30 M x 64: 4.65 vs 5.8-6.4 ms; 3 M rows: equal; below that
    // the small-batch kernel's one-launch dump mode wins (1 M x 64: 0.32 vs 0.38 ms).  At 100 M rows the batched kernel's
    // HBM rate is erratic (128 queries: 15.1 .. 21.0 ms over four runs; 17 / 32 / 64 queries 16.6 / 17.9 / 18.3 ms against
    // 15.1-15.8 / ~16 / 17.2-18.1 ms on the small-batch kernel), so the hand-off at 17 queries applies up to 50 M rows.
    const bool mid_shard = idx->ntotal > 3500000 && idx->ntotal <= 50000000;
    const int small_dflt = idx->dpad > kMaxKBlocks * kKBlock ? 128 : (mid_shard ? 16 : 64);
    const int small_max = env_int("IVR_MMA_SMALL_MAX_NQ", small_dflt);
    // beyond 1024 dims only the small-batch kernel exists (its query tile loops over any number of k-blocks)
    if (mode == 3 || ((mode == 0 || !mma_supported(idx, nq, k)) && nq <= small_max && mma_small_supported(idx, nq, k)))
        return search_mma_small(idx, q_dev, nq, k, D_dev, I_dev, id_offset, st);
    if (!mma_supported(idx, nq, k)) {
        set_error("search_mma: dim=%d with %lld queries fits no tcgen05 kernel", idx->dim, static_cast<long long>(nq));
        return IVR_EUNSUPPORTED;
    }
    // measured (k=100, seeded launches): 4096 queries -- 3 M rows 11.6 ms query-tile-resident vs 11.5 ms
    // row-tile-resident, 10 M 38.7 vs 34.0, 100 M 405 vs 325; 1024 queries -- 10 M 8.4 vs 9.6.  The
    // row-tile-resident kernel moves 9x fewer bytes (the GPU is power-capped) but spreads a query over more
    // candidate lists: it takes over from 2048 queries on >= 3 M rows and from 4 query tiles on >= 12 M rows
    const bool wide = idx->dpad > kMaxKBlocks * kKBlock;           // 513..1024 dims: only the row-tile-resident kernel fits
    const int64_t xres_min_rows = static_cast<int64_t>(env_int("IVR_MMA_XRES_MIN_ROWS_M", nq >= 2048 ? 3 : 12)) * 1000000;
    const bool xres = wide || (mode == 2) || (mode == 0 && nq > 3 * kTileQ * 2 && idx->ntotal >= xres_min_rows);
    // per launch: row-tile-resident is bounded by its candidate-list workspace, query-tile-resident by
    // one query tile per CTA group
    idx->last_kernel = xres ? "search_mma_xres_kernel" : "search_mma_kernel";
    int64_t per_launch = static_cast<int64_t>(idx->sm_count / cg) * kTileQ * cg;
    if (xres) {                                                    // one list per (pair, set, query): keep them under 8 GiB
        const int64_t per_query = static_cast<int64_t>(idx->sm_count / 2) * 2 * (2 * kcap_for(k)) * 8;
        per_launch = std::min<int64_t>(16384, std::max<int64_t>(2 * kTileQ, ((8ll << 30) / per_query) / (2 * kTileQ) * (2 * kTileQ)));
    }
    for (int64_t q0 = 0; q0 < nq; q0 += per_launch) {
        const int64_t b = std::min(per_launch, nq - q0);
        IVR_TRY(search_mma_batch(idx, q_dev + q0 * idx->dim, b, k, D_dev ? D_dev + q0 * k : nullptr, I_dev + q0 * k, id_offset, st,
                                 cg, xres, q0 == 0));
    }
    return IVR_OK;
}

}  // namespace ivr

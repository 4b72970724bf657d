// topk_merge.cu -- K5: exact k-way merge of candidate lists (one CTA per query).
//
// Used (a) after the streaming / MMA scoring kernels to fold the per-warp or
// per-CTA partial lists into the final [nq,k] result, and (b) after the NCCL
// all-gather of the row shards' local top-k (ivr_topk_merge_device).
//
// Method: MSB-first radix select on the 64-bit candidate keys (8 bits per pass,
// shared-memory histogram) finds the k-th largest key exactly, the k survivors
// are gathered into shared memory and bitonic-sorted.  Integer-exact; ties on
// score resolve to the lower row id because the id is part of the key.
#include "index.cuh"

#include <algorithm>
#include <type_traits>

namespace ivr {

constexpr int kMergeThreads = 256;
// Lists folded by one CTA in a non-final level.  A CTA that holds the list lengths in shared memory (<= kFlatLists
// lists) fetches every candidate through a flattened index, so a wide fan-in costs no dependent-load chain: the 148
// lists per query of the row-tile-resident kernel fold in ONE level -- wherever the batch alone keeps the machine full
// of CTAs.  Few queries x many lists (the small-batch kernel: 592 lists for <= 128 queries) keep the narrow fan-in: they
// need the CTAs of the first level.
static int merge_fan_in(int k, int64_t nq, int n_lists) {
    const int64_t ctas_wide = nq * ((n_lists + 255) / 256);
    return (k <= 128 && ctas_wide >= 1024) ? 256 : 64;
}
constexpr int kStageCap  = 2048;      // keys of one (query, list group) staged in shared memory (16 KB)
constexpr int kFlatLists = 256;       // most lists per CTA on the flattened path (= kMergeThreads: one length per thread)

static int kpad_for(int k) { int p = 2; while (p < k) p <<= 1; return p; }

struct MergeOut {
    float*    D;            // final
    int64_t*  I;
    int64_t   id_offset;
    const float* q_scale;   // final: per-query score multiplier (nullptr = 1)
    uint64_t* entries;      // non-final: [groups, nq, k]
    int*      counts;       // non-final: [groups, nq]
    int64_t   nq;
};

// key of a materialised score; 0 (no key) for NaN, the score of a row holding a NaN, which is never returned
__device__ __forceinline__ uint64_t dense_key(float score, int64_t row) {
    return isnan(score) ? 0ull : make_key(score, static_cast<uint32_t>(row));
}

template <typename F>
__device__ __forceinline__ void for_each_key(const MergeIn& in, int64_t q, int l0, int l1, F&& f) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    if (in.dense) {                                  // materialised scores: rows l * dense_len + i
        const float* base = in.dense + q * in.dense_q_stride;
        for (int l = l0 + warp; l < l1; l += nwarps)
            for (int i = lane; i < in.dense_len; i += 32) {
                const int64_t row = static_cast<int64_t>(l) * in.dense_len + i;
                const uint64_t key = (row < in.dense_rows) ? dense_key(base[row], row) : 0ull;
                if (key != 0ull) f(key);
            }
        return;
    }
    for (int l = l0 + warp; l < l1; l += nwarps) {
        const int cnt = in.counts ? in.counts[l * in.cnt_list_stride + q * in.cnt_q_stride]
                                  : in.fixed_count;
        const uint64_t* base = in.entries + l * in.list_stride +
                               (in.interleave ? (q >> 5) * in.q_stride * 32 + (q & 31) : q * in.q_stride);
        const int es = in.interleave ? 32 : 1;
        for (int i = lane; i < cnt; i += 32) {
            uint64_t key = base[static_cast<int64_t>(i) * es];
            if (in.raw) key = make_key(__uint_as_float(static_cast<uint32_t>(key)), static_cast<uint32_t>(key >> 32));
            if (key != 0ull) f(key);
        }
    }
}

// shared-memory bitonic sort, DESCENDING, of n (a power of two) keys; ends with a barrier
__device__ __forceinline__ void block_bitonic_desc(uint64_t* s_keys, int n) {
    for (int s = 2; s <= n; s <<= 1) {
        for (int t = s >> 1; t > 0; t >>= 1) {
            for (int i = threadIdx.x; i < (n >> 1); i += blockDim.x) {
                const int lo = 2 * i - (i & (t - 1));
                const int hi = lo + t;
                const bool desc = (lo & s) == 0;
                const uint64_t a = s_keys[lo], b = s_keys[hi];
                if ((a < b) == desc) { s_keys[lo] = b; s_keys[hi] = a; }
            }
            __syncthreads();
        }
    }
}

struct MergeShared {
    int      hist[256];
    uint64_t prefix, mask;
    int      remaining, done, n, neq, total;
    int      off[kFlatLists + 1];       // flattened path: exclusive prefix sum of the list lengths
    int      wsum[kMergeThreads / 32];
};

// k-th-largest search, one 8-bit digit: warp 0 scans the 256-bin histogram from the top bin down (32 bins per step,
// shuffle prefix sums) and publishes the digit, the rank that remains inside its bin and whether the whole bin is
// needed (then the select is finished).  Call with the histogram complete (after a barrier); ends with a barrier.
__device__ __forceinline__ void radix_scan_bins(MergeShared& sh, uint64_t prefix, uint64_t mask, int remaining, int shift) {
    const int tid = threadIdx.x, lane = tid & 31;
    if (tid < 32) {
        int cum_before = 0, found = 0, rem_after = remaining;
        bool hit_any = false;
        for (int base = 224; base >= 0 && !hit_any; base -= 32) {
            const int c = sh.hist[base + 31 - lane];                 // lane 0 holds the highest bin of the group
            int incl = c;
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
            const unsigned hit = __ballot_sync(0xffffffffu, cum_before + incl >= remaining);
            if (hit) {
                const int l0 = __ffs(hit) - 1;
                found = base + 31 - l0;
                rem_after = remaining - (cum_before + __shfl_sync(0xffffffffu, incl - c, l0));
                hit_any = true;
            }
            cum_before += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) {                                             // fewer than `remaining` keys match: bin 0 takes the rest
            if (!hit_any) { found = 0; rem_after = remaining - (cum_before - sh.hist[0]); }
            sh.remaining = rem_after;
            sh.prefix = prefix | (static_cast<uint64_t>(found) << shift);
            sh.mask = mask | (0xffull << shift);
            sh.done = (sh.hist[found] == rem_after);                 // the whole bin is needed: stop early
        }
    }
    __syncthreads();
}

// The k best keys are in s_keys[0 .. kpad) in any order (0-padded): sort them descending.  Up to 256 slots one warp
// sorts them in registers (no block barrier per network stage); larger k uses the block-wide network.
__device__ __forceinline__ void sort_result(uint64_t* s_keys, int kpad) {
    __syncthreads();
    if (kpad > 256) { block_bitonic_desc(s_keys, kpad); return; }
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        auto run = [&](auto tag) {
            constexpr int E = decltype(tag)::value;
            uint64_t v[E];
#pragma unroll
            for (int j = 0; j < E; ++j) { const int g = lane * E + j; v[j] = g < kpad ? s_keys[g] : 0ull; }
            warp_sort_desc<E>(v, lane);
#pragma unroll
            for (int j = 0; j < E; ++j) { const int g = lane * E + j; if (g < kpad) s_keys[g] = v[j]; }
        };
        if (kpad <= 32) run(std::integral_constant<int, 1>{});
        else if (kpad <= 64) run(std::integral_constant<int, 2>{});
        else if (kpad <= 128) run(std::integral_constant<int, 4>{});
        else run(std::integral_constant<int, 8>{});
    }
    __syncthreads();
}

// Flattened path of block_select_sort (<= kFlatLists lists, not dense).  The in-place select further down walks the
// lists once per radix pass, one list per warp step, every step a dependent pair of global loads (length, then
// entries): ~20 steps x 2 round trips x up to 10 passes per CTA.  Here the lengths are fetched with ONE load per thread
// and prefix-summed in shared memory; candidate idx of the group is then addressed directly (binary search of its list
// in the prefix sums), so all loads of a pass are independent.  Up to kStageCap candidates are fetched once into shared
// memory (STAGED) and every radix pass runs there; larger groups re-read global memory through the same flattened index.
// The k-th largest key is found digit by digit (8 bits, shared histogram, warp-parallel bin scan), the survivors are
// compacted into s_keys[0 .. kpad) and sorted by one warp.
template <bool STAGED>
__device__ __forceinline__ uint64_t flat_key(const MergeIn& in, int64_t q, int l0, int n_l, int idx,
                                             const uint64_t* stage, const MergeShared& sh) {
    if (STAGED) return stage[idx];
    int lo = 0, hi = n_l;                                // off[] is non-decreasing: the last list with off <= idx is
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (sh.off[mid] <= idx) lo = mid; else hi = mid; }   // non-empty
    const uint64_t* base = in.entries + (l0 + lo) * in.list_stride +
                           (in.interleave ? (q >> 5) * in.q_stride * 32 + (q & 31) : q * in.q_stride);
    uint64_t key = base[static_cast<int64_t>(idx - sh.off[lo]) * (in.interleave ? 32 : 1)];
    if (in.raw) key = make_key(__uint_as_float(static_cast<uint32_t>(key)), static_cast<uint32_t>(key >> 32));
    return key;
}

template <bool STAGED>
__device__ int flat_select(const MergeIn& in, int64_t q, int l0, int n_l, int total, int k, int kpad, uint64_t* s_keys,
                           const uint64_t* stage, MergeShared& sh) {
    const int tid = threadIdx.x;
    uint64_t prefix = 0, mask = 0;
    int remaining = k;
    for (int pass = 0; pass < 8; ++pass) {
        const int shift = 56 - 8 * pass;
        sh.hist[tid] = 0;                                // kMergeThreads == 256 bins
        __syncthreads();
        for (int idx = tid; idx < total; idx += kMergeThreads) {
            const uint64_t key = flat_key<STAGED>(in, q, l0, n_l, idx, stage, sh);
            if ((key & mask) == prefix) atomicAdd(&sh.hist[(key >> shift) & 0xff], 1);
        }
        __syncthreads();
        radix_scan_bins(sh, prefix, mask, remaining, shift);
        prefix = sh.prefix; mask = sh.mask; remaining = sh.remaining;
        if (sh.done) break;
    }
    // keys above the k-th digit string are in; of the keys equal to it, `remaining` (all of them when the bin was
    // needed whole; any `remaining` of them otherwise -- they can differ only below the bits examined, i.e. not at all
    // after 8 passes)
    int zeros = 0;
    for (int idx = tid; idx < total; idx += kMergeThreads) {
        const uint64_t key = flat_key<STAGED>(in, q, l0, n_l, idx, stage, sh);
        zeros += key == 0ull;
        const uint64_t km = key & mask;
        if (km > prefix) {
            s_keys[atomicAdd(&sh.n, 1)] = key;
        } else if (km == prefix) {
            const int e = atomicAdd(&sh.neq, 1);
            if (e < remaining) s_keys[k - remaining + e] = key;      // tail slots, disjoint from the > slots
        }
    }
    for (int o = 16; o > 0; o >>= 1) zeros += __shfl_xor_sync(0xffffffffu, zeros, o);
    if ((tid & 31) == 0 && zeros) atomicAdd(&sh.total, zeros);       // sh.total counts the padding keys here
    sort_result(s_keys, kpad);
    return min(total - sh.total, k);
}

// Returns -1 when the group does not qualify (dense input, > kFlatLists lists).  s_keys holds kpad + kStageCap keys.
__device__ int block_flat_select_sort(const MergeIn& in, int64_t q, int l0, int l1, int k, int kpad, uint64_t* s_keys,
                                      MergeShared& sh) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_l = l1 - l0;
    if (in.dense || n_l > kFlatLists || blockDim.x != kMergeThreads) return -1;
    // list lengths -> exclusive prefix sum (one length per thread)
    int c = 0;
    if (tid < n_l) c = in.counts ? in.counts[(l0 + tid) * in.cnt_list_stride + q * in.cnt_q_stride] : in.fixed_count;
    int incl = c;
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) sh.wsum[warp] = incl;
    if (tid == 0) { sh.total = 0; sh.n = 0; sh.neq = 0; }
    for (int i = tid; i < kpad; i += kMergeThreads) s_keys[i] = 0ull;
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < kMergeThreads / 32; ++w) { const int v = sh.wsum[w]; if (w < warp) before += v; total += v; }
    sh.off[tid] = before + incl - c;
    uint64_t* stage = s_keys + kpad;
    __syncthreads();
    if (total <= kpad) {                                 // everything survives: fetch straight into the result slots
        int zeros = 0;
        for (int idx = tid; idx < total; idx += kMergeThreads) {
            const uint64_t key = flat_key<false>(in, q, l0, n_l, idx, stage, sh);
            zeros += key == 0ull;
            s_keys[idx] = key;
        }
        for (int o = 16; o > 0; o >>= 1) zeros += __shfl_xor_sync(0xffffffffu, zeros, o);
        if (lane == 0 && zeros) atomicAdd(&sh.total, zeros);
        sort_result(s_keys, kpad);
        return min(total - sh.total, k);
    }
    if (total <= kStageCap) {
        for (int idx = tid; idx < total; idx += kMergeThreads) stage[idx] = flat_key<false>(in, q, l0, n_l, idx, stage, sh);
        __syncthreads();
        return flat_select<true>(in, q, l0, n_l, total, k, kpad, s_keys, stage, sh);
    }
    return flat_select<false>(in, q, l0, n_l, total, k, kpad, s_keys, stage, sh);
}

// Block-level exact selection: the (at most) k largest keys of lists [l0, l1) of query q, sorted descending in
// s_keys[0 .. kpad) (0-padded).  Returns the number of valid entries.  MSB-first 8-bit radix select on the 64-bit
// keys, then a sort of the survivors.  Every thread of the block must call it.
__device__ int block_select_sort(const MergeIn& in, int64_t q, int l0, int l1, int k, int kpad, uint64_t* s_keys,
                                 MergeShared& sh) {
    const int tid = threadIdx.x;
    {
        const int flat = block_flat_select_sort(in, q, l0, l1, k, kpad, s_keys, sh);
        if (flat >= 0) return flat;
    }
    // in-place select: dense input (materialised scores) or more than kFlatLists lists
    if (tid == 0) { sh.total = 0; sh.n = 0; sh.neq = 0; sh.prefix = 0; sh.mask = 0; sh.remaining = k; sh.done = 0; }
    for (int i = tid; i < kpad; i += blockDim.x) s_keys[i] = 0ull;
    __syncthreads();

    {   // total number of real candidates
        int local = 0;
        for_each_key(in, q, l0, l1, [&](uint64_t) { ++local; });
        for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
        if ((tid & 31) == 0 && local) atomicAdd(&sh.total, local);
    }
    __syncthreads();
    const int total = sh.total;

    if (total <= k) {
        for_each_key(in, q, l0, l1, [&](uint64_t key) { s_keys[atomicAdd(&sh.n, 1)] = key; });
    } else {
        uint64_t prefix = 0, mask = 0;
        int remaining = k;
        for (int pass = 0; pass < 8; ++pass) {
            const int shift = 56 - 8 * pass;
            for (int i = tid; i < 256; i += blockDim.x) sh.hist[i] = 0;
            __syncthreads();
            for_each_key(in, q, l0, l1, [&](uint64_t key) {
                if ((key & mask) == prefix) atomicAdd(&sh.hist[(key >> shift) & 0xff], 1);
            });
            __syncthreads();
            radix_scan_bins(sh, prefix, mask, remaining, shift);
            prefix = sh.prefix; mask = sh.mask; remaining = sh.remaining;
            if (sh.done) break;
        }
        for_each_key(in, q, l0, l1, [&](uint64_t key) {
            const uint64_t km = key & mask;
            if (km > prefix) {
                s_keys[atomicAdd(&sh.n, 1)] = key;
            } else if (km == prefix) {
                const int e = atomicAdd(&sh.neq, 1);
                if (e < remaining) s_keys[k - remaining + e] = key;   // tail slots, disjoint from the > slots
            }
        });
    }
    sort_result(s_keys, kpad);
    return min(total, k);
}

// final output of one query from its sorted keys: (D, I) rows, or packed keys when D == nullptr
__device__ __forceinline__ void write_final(const MergeOut& out, int64_t q, int k, const uint64_t* s_keys, int nvalid) {
    const int tid = threadIdx.x;
    const float scale = out.q_scale ? out.q_scale[q] : 1.0f;
    if (out.D == nullptr) {
        // packed-key output for the cross-shard exchange: final score, 32-bit GLOBAL row id, 0 = padding
        uint64_t* K = reinterpret_cast<uint64_t*>(out.I);
        const uint32_t off = static_cast<uint32_t>(out.id_offset);
        for (int i = tid; i < k; i += blockDim.x) {
            const uint64_t key = s_keys[i];
            K[q * k + i] = (i < nvalid) ? make_key(key_score(key) * scale, key_row(key) + off) : 0ull;
        }
        return;
    }
    for (int i = tid; i < k; i += blockDim.x) {
        const uint64_t key = s_keys[i];
        const bool ok = i < nvalid;
        out.D[q * k + i] = ok ? key_score(key) * scale : -3.402823466e+38f;
        out.I[q * k + i] = ok ? static_cast<int64_t>(key_row(key)) + out.id_offset : -1;
    }
}

template <bool FINAL>
__global__ void __launch_bounds__(kMergeThreads)
merge_kernel(MergeIn in, MergeOut out, int lists_per_group, int k, int kpad) {
    extern __shared__ uint64_t s_keys[];               // kpad
    __shared__ MergeShared sh;
    const int64_t q = blockIdx.x;
    const int grp = blockIdx.y;
    const int l0 = grp * lists_per_group;
    const int l1 = min(l0 + lists_per_group, in.n_lists);
    const int tid = threadIdx.x;
    const int nvalid = block_select_sort(in, q, l0, l1, k, kpad, s_keys, sh);
    if (FINAL) {
        write_final(out, q, k, s_keys, nvalid);
    } else {
        uint64_t* dst = out.entries + (static_cast<int64_t>(grp) * out.nq + q) * k;
        for (int i = tid; i < k; i += blockDim.x) dst[i] = (i < nvalid) ? s_keys[i] : 0ull;
        if (tid == 0) out.counts[static_cast<int64_t>(grp) * out.nq + q] = nvalid;
    }
}

// ---------------------------------------------------------------------------
// One-launch merge for MANY short lists (the streaming kernel leaves 2368 per-warp lists per query).
//
// Bound from the list maxima: the k-th largest of the per-list MAXIMUM scores, T, is reached by k distinct rows, so the
// final k-th best is >= T and every row of the final top-k has score >= T.  The rows are dealt to the warps round-robin
// (search_stream.cu), so the best rows sit in different lists and T lands within a few ranks of the true k-th best: only
// ~k of the ~10^5 .. 10^6 listed candidates survive the filter "score >= T".
//   1. every CTA finds T from the maxima (32-bit radix select in shared memory; redundant but parallel and L2-fed);
//   2. the CTAs split the lists and append the survivors to one pool per query (warp-aggregated atomic);
//   3. the LAST CTA to finish (ticket) sorts the pool and writes the result.  If the pool overflowed (rows clustered
//      in few lists, massive ties) it falls back to the exact radix select over all lists -- slow but always correct.
// The ticket and the pool counter are reset by the last CTA: self-cleaning between calls (zeroed once by the caller).
// ---------------------------------------------------------------------------
struct SelectArgs {
    const uint32_t* maxima;     // [n_lists * cnt_list_stride ...] ordered-score maximum of every list (same strides as counts)
    // the values the bound T is searched in: maximum g of query q at tmax[g * t_stride_g + q * t_stride_q], g < n_t.
    // Either the list maxima themselves, or the maxima of <= 1024 GROUPS of consecutive lists (dense mode: ~10^4 .. 10^5
    // tiles per query would make the redundant per-CTA search the dominant cost; ~1000 groups bound just as tightly).
    const uint32_t* tmax;
    int64_t   t_stride_g, t_stride_q;
    int       n_t;
    uint64_t* pool;             // [nq][pool_cap]
    int*      pool_cnt;         // [nq]
    int*      ticket;           // [nq]
    int       pool_cap;         // power of two
};

__global__ void __launch_bounds__(kMergeThreads)
merge_select_kernel(MergeIn in, MergeOut out, SelectArgs sa, int k, int kpad) {
    extern __shared__ uint64_t s_keys[];               // max(kpad, pool_cap)
    __shared__ MergeShared sh;
    __shared__ uint32_t s_T;
    __shared__ int s_last;
    const int64_t q = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int M = in.n_lists;

    // ---- 1. T = k-th largest (group) maximum (0 when fewer than k of them are set: admit everything) ----
    {
        // the maxima are fetched ONCE, all loads of a thread in flight together (up to 16 per thread = 4096 values:
        // 2368 lists of the streaming kernel, <= 1024 tile groups in dense mode); the four radix passes then run on
        // registers -- a dependent global load per value and pass used to be most of this kernel's 21 us
        constexpr int kMine = 16;
        uint32_t mine[kMine];
        const bool in_regs = sa.n_t <= kMine * kMergeThreads;
        if (in_regs) {
#pragma unroll
            for (int j = 0; j < kMine; ++j) {
                const int g = tid + j * kMergeThreads;
                mine[j] = (g < sa.n_t) ? sa.tmax[g * sa.t_stride_g + q * sa.t_stride_q] : 0u;
            }
        }
        uint32_t prefix = 0, mask = 0;
        int remaining = k;
        for (int pass = 0; pass < 4; ++pass) {
            const int shift = 24 - 8 * pass;
            for (int i = tid; i < 256; i += blockDim.x) sh.hist[i] = 0;
            __syncthreads();
            if (in_regs) {
#pragma unroll
                for (int j = 0; j < kMine; ++j)
                    if (tid + j * kMergeThreads < sa.n_t && (mine[j] & mask) == prefix)
                        atomicAdd(&sh.hist[(mine[j] >> shift) & 0xff], 1);
            } else {
                for (int g = tid; g < sa.n_t; g += blockDim.x) {
                    const uint32_t v = sa.tmax[g * sa.t_stride_g + q * sa.t_stride_q];
                    if ((v & mask) == prefix) atomicAdd(&sh.hist[(v >> shift) & 0xff], 1);
                }
            }
            __syncthreads();
            if (warp == 0) {                             // warp-parallel scan from the top bin down
                int cum_before = 0, found = -1, rem_after = remaining;
                for (int base = 224; base >= 0 && found < 0; base -= 32) {
                    const int c = sh.hist[base + 31 - lane];             // lane 0 holds the highest bin of the group
                    int incl = c;
                    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
                    const unsigned hit = __ballot_sync(0xffffffffu, cum_before + incl >= remaining);
                    if (hit) {
                        const int l0 = __ffs(hit) - 1;
                        found = base + 31 - l0;
                        rem_after = remaining - (cum_before + __shfl_sync(0xffffffffu, incl - c, l0));
                    }
                    cum_before += __shfl_sync(0xffffffffu, incl, 31);
                }
                if (lane == 0) {
                    if (found < 0) { sh.done = 2; }      // fewer than `remaining` maxima match: not enough lists
                    else {
                        sh.prefix = prefix | (static_cast<uint32_t>(found) << shift);
                        sh.mask = mask | (0xffu << shift);
                        sh.remaining = rem_after;
                        sh.done = 0;
                    }
                }
            }
            __syncthreads();
            if (sh.done == 2) break;
            prefix = static_cast<uint32_t>(sh.prefix); mask = static_cast<uint32_t>(sh.mask); remaining = sh.remaining;
        }
        if (tid == 0) s_T = (sh.done == 2) ? 0u : prefix;
        __syncthreads();
    }
    const uint32_t T = s_T;

    // ---- 2. filter this CTA's share of the lists into the pool ----
    uint64_t* pool = sa.pool + q * sa.pool_cap;
    const int per = (M + gridDim.x - 1) / gridDim.x;
    const int l0 = blockIdx.x * per, l1 = min(l0 + per, M);
    for (int lb = l0 + warp * 32; lb < l1; lb += nwarps * 32) {      // 32 lists per step: one maximum per lane
        const int lmine = lb + lane;
        unsigned todo = __ballot_sync(0xffffffffu, lmine < l1 &&
                                      sa.maxima[lmine * in.cnt_list_stride + q * in.cnt_q_stride] >= T);
        while (todo) {                                               // lists with a maximum below T cannot contribute
            const int l = lb + __ffs(todo) - 1;
            todo &= todo - 1;
            const int cnt = in.dense ? in.dense_len
                                     : (in.counts ? in.counts[l * in.cnt_list_stride + q * in.cnt_q_stride] : in.fixed_count);
            const uint64_t* base = in.dense ? nullptr : in.entries + l * in.list_stride +
                                   (in.interleave ? (q >> 5) * in.q_stride * 32 + (q & 31) : q * in.q_stride);
            const int es = in.interleave ? 32 : 1;
            for (int i0 = 0; i0 < cnt; i0 += 32 * 8) {               // 8 entries per lane in flight: one load latency per 256 entries
                uint64_t key[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int i = i0 + u * 32 + lane;
                    key[u] = 0ull;
                    if (in.dense) {
                        const int64_t row = static_cast<int64_t>(l) * in.dense_len + i;
                        if (i < cnt && row < in.dense_rows)
                            key[u] = dense_key(in.dense[q * in.dense_q_stride + row], row);
                    } else if (i < cnt) {
                        key[u] = base[static_cast<int64_t>(i) * es];
                        if (in.raw) key[u] = make_key(__uint_as_float(static_cast<uint32_t>(key[u])), static_cast<uint32_t>(key[u] >> 32));
                    }
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const bool keep = key[u] != 0ull && static_cast<uint32_t>(key[u] >> 32) >= T;
                    const unsigned m = __ballot_sync(0xffffffffu, keep);
                    if (m) {
                        int pos = 0;
                        if (lane == 0) pos = atomicAdd(sa.pool_cnt + q, __popc(m));
                        pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(m & ((1u << lane) - 1u));
                        if (keep && pos < sa.pool_cap) pool[pos] = key[u];
                    }
                }
            }
        }
    }

    // ---- 3. last CTA: sort the pool (or fall back to the exact select) and write the result ----
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(sa.ticket + q, 1) == static_cast<int>(gridDim.x) - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int n_pool = *reinterpret_cast<volatile int*>(sa.pool_cnt + q);
    int nvalid;
    if (n_pool <= sa.pool_cap) {
        int np2 = kpad;                                  // sort size: power of two >= max(n_pool, k)
        while (np2 < n_pool) np2 <<= 1;
        for (int i = tid; i < np2; i += blockDim.x) s_keys[i] = (i < n_pool) ? __ldcg(pool + i) : 0ull;
        __syncthreads();
        block_bitonic_desc(s_keys, np2);
        nvalid = min(n_pool, k);
    } else {
        nvalid = block_select_sort(in, q, 0, M, k, kpad, s_keys, sh);
    }
    write_final(out, q, k, s_keys, nvalid);
    if (tid == 0) { sa.pool_cnt[q] = 0; sa.ticket[q] = 0; }
}


size_t merge_tmp_entries(int n_lists, int64_t nq, int k) {
    // levels shrink by the fan-in; two ping-pong buffers sized for the first level
    const int fan = merge_fan_in(k, nq, n_lists);
    if (n_lists <= fan) return 0;
    const int64_t g1 = (n_lists + fan - 1) / fan;
    const int64_t g2 = (g1 + fan - 1) / fan;
    return static_cast<size_t>((g1 + g2) * nq * k);
}

int merge_lists_final(const MergeIn& in0, int64_t nq, int k, float* D_dev, int64_t* I_dev,
                      int64_t id_offset, uint64_t* tmp_entries, int* tmp_counts,
                      cudaStream_t st, int* n_launches, const float* q_scale) {
    if (nq <= 0) return IVR_OK;
    const int kpad = kpad_for(k);
    const size_t smem = static_cast<size_t>(kpad + kStageCap) * sizeof(uint64_t);
    const int kMergeFanIn = merge_fan_in(k, nq, in0.n_lists);
    MergeIn in = in0;
    int level = 0;
    uint64_t* ebuf = tmp_entries;
    int*      cbuf = tmp_counts;
    while (in.n_lists > kMergeFanIn) {
        const int groups = (in.n_lists + kMergeFanIn - 1) / kMergeFanIn;
        if (!ebuf || !cbuf) { set_error("merge: scratch missing for %d lists", in.n_lists); return IVR_EINVAL; }
        MergeOut out{};
        out.entries = ebuf; out.counts = cbuf; out.nq = nq;
        dim3 grid(static_cast<unsigned>(nq), static_cast<unsigned>(groups));
        merge_kernel<false><<<grid, kMergeThreads, smem, st>>>(in, out, kMergeFanIn, k, kpad);
        IVR_CUDA(cudaGetLastError());
        if (n_launches) ++*n_launches;
        MergeIn nx{};
        nx.entries = ebuf; nx.counts = cbuf;
        nx.list_stride = nq * k; nx.q_stride = k;
        nx.cnt_list_stride = nq; nx.cnt_q_stride = 1;
        nx.n_lists = groups; nx.fixed_count = 0; nx.raw = 0;
        ebuf += static_cast<size_t>(groups) * nq * k;
        cbuf += static_cast<size_t>(groups) * nq;
        in = nx;
        if (++level > 4) { set_error("merge: too many levels"); return IVR_EINVAL; }
    }
    MergeOut out{};
    out.D = D_dev; out.I = I_dev; out.id_offset = id_offset; out.nq = nq; out.q_scale = q_scale;
    dim3 grid(static_cast<unsigned>(nq), 1);
    merge_kernel<true><<<grid, kMergeThreads, smem, st>>>(in, out, in.n_lists, k, kpad);
    IVR_CUDA(cudaGetLastError());
    if (n_launches) ++*n_launches;
    return IVR_OK;
}

// One-launch merge by the list-maxima bound (see merge_select_kernel).  `maxima` uses the strides of in.counts;
// `pool` holds nq * kSelectPoolCap keys, `pool_cnt` / `ticket` nq ints each, all zero on entry (the kernel re-zeroes them).
int merge_select_final(const MergeIn& in, const uint32_t* maxima, int64_t nq, int k, float* D_dev, int64_t* I_dev,
                       int64_t id_offset, uint64_t* pool, int* pool_cnt, int* ticket, int sm_count, cudaStream_t st,
                       int* n_launches, const float* q_scale, const uint32_t* group_max, int n_groups) {
    if (nq <= 0) return IVR_OK;
    if (k > kSelectMaxK || nq > 65535) { set_error("merge_select: k=%d / nq=%lld outside its range", k, static_cast<long long>(nq)); return IVR_EINVAL; }
    const int kpad = kpad_for(k);
    const size_t smem = static_cast<size_t>(std::max(kpad, kSelectPoolCap)) * sizeof(uint64_t);
    MergeOut out{};
    out.D = D_dev; out.I = I_dev; out.id_offset = id_offset; out.nq = nq; out.q_scale = q_scale;
    SelectArgs sa{};
    sa.maxima = maxima; sa.pool = pool; sa.pool_cnt = pool_cnt; sa.ticket = ticket; sa.pool_cap = kSelectPoolCap;
    if (group_max) { sa.tmax = group_max; sa.t_stride_g = 1; sa.t_stride_q = n_groups; sa.n_t = n_groups; }
    else { sa.tmax = maxima; sa.t_stride_g = in.cnt_list_stride; sa.t_stride_q = in.cnt_q_stride; sa.n_t = in.n_lists; }
    // enough CTAs that the filter pass is spread over the machine, few enough that the redundant T search stays cheap
    const int ctas = std::max(1, std::min(in.n_lists / 16, std::max(1, 2 * sm_count / static_cast<int>(std::min<int64_t>(nq, 2 * sm_count)))));
    dim3 grid(static_cast<unsigned>(ctas), static_cast<unsigned>(nq));
    merge_select_kernel<<<grid, kMergeThreads, smem, st>>>(in, out, sa, k, kpad);
    IVR_CUDA(cudaGetLastError());
    if (n_launches) ++*n_launches;
    return IVR_OK;
}

// Same reduction, but the result stays in key form: out_keys [nq, k] (descending, 0-padded) and
// out_counts [nq].  Used between the two phases of the batched search.
int merge_lists_keys(const MergeIn& in0, int64_t nq, int k, uint64_t* out_keys, int* out_counts,
                     uint64_t* tmp_entries, int* tmp_counts, cudaStream_t st, int* n_launches) {
    if (nq <= 0) return IVR_OK;
    const int kpad = kpad_for(k);
    const size_t smem = static_cast<size_t>(kpad + kStageCap) * sizeof(uint64_t);
    const int kMergeFanIn = merge_fan_in(k, nq, in0.n_lists);
    MergeIn in = in0;
    uint64_t* ebuf = tmp_entries;
    int*      cbuf = tmp_counts;
    for (int level = 0; ; ++level) {
        const bool last = in.n_lists <= kMergeFanIn;
        const int groups = last ? 1 : (in.n_lists + kMergeFanIn - 1) / kMergeFanIn;
        if (!last && (!ebuf || !cbuf)) { set_error("merge: scratch missing for %d lists", in.n_lists); return IVR_EINVAL; }
        MergeOut out{};
        out.entries = last ? out_keys : ebuf; out.counts = last ? out_counts : cbuf; out.nq = nq;
        dim3 grid(static_cast<unsigned>(nq), static_cast<unsigned>(groups));
        merge_kernel<false><<<grid, kMergeThreads, smem, st>>>(in, out, last ? in.n_lists : kMergeFanIn, k, kpad);
        IVR_CUDA(cudaGetLastError());
        if (n_launches) ++*n_launches;
        if (last) return IVR_OK;
        MergeIn nx{};
        nx.entries = ebuf; nx.counts = cbuf;
        nx.list_stride = nq * k; nx.q_stride = k;
        nx.cnt_list_stride = nq; nx.cnt_q_stride = 1;
        nx.n_lists = groups; nx.fixed_count = 0; nx.raw = 0;
        ebuf += static_cast<size_t>(groups) * nq * k;
        cbuf += static_cast<size_t>(groups) * nq;
        in = nx;
        if (level > 4) { set_error("merge: too many levels"); return IVR_EINVAL; }
    }
}

// ---------------------------------------------------------------------------
// (D, I) shard lists -> packed keys, for the post-all-gather merge.  The key holds a 32-bit row id:
// ids at or above 2^32 cannot be represented and raise the flag (the caller rejects the merge).
// ---------------------------------------------------------------------------
__global__ void pack_parts_kernel(const float* __restrict__ D, const int64_t* __restrict__ I,
                                  uint64_t* __restrict__ keys, int64_t n) {
    const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (i >= n) return;
    const int64_t id = I[i];
    keys[i] = (id < 0 || id > 0xffffffffll) ? 0ull : make_key(D[i], static_cast<uint32_t>(id));
}

int pack_parts(const float* D, const int64_t* I, uint64_t* keys, int64_t n, cudaStream_t st) {
    if (n <= 0) return IVR_OK;
    const int threads = 256;
    const int64_t blocks = (n + threads - 1) / threads;
    pack_parts_kernel<<<static_cast<unsigned>(blocks), threads, 0, st>>>(D, I, keys, n);
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

}  // namespace ivr

// range_search.cu -- exact range search: every stored row whose inner product with a query is > radius.
//
// Replaces lims, D, I = index.range_search(x, radius) of faiss.IndexFlatIP (not called by the reference).
//   1. queries -> fp16, scaled by a power of two (launch_queries_to_f16), one chunk of <= small_range_chunk() queries
//      at a time;
//   2. one K1s launch per chunk in RANGE mode (search_mma_small.cu): every hit goes to one pool of
//      (packed key, query) pairs; the 64-bit cursor counts every hit, also those past the pool's capacity;
//   3. if the pool held them all: histogram by query, exclusive scan into lims, scatter into the query segments,
//      segmented sort descending (the key order: score descending, then lower row), unpack to D / I.
// Step 3 reads the cursor on the device, so nothing here waits for the GPU.  A filtered search (ivr_selection) runs
// step 2 on search_mma_small_sel_range_kernel over the row tiles of a cut of the selection only (SelCut: all stored rows,
// or a search window's).  The self-join (range_self_join_device)
// fills the same pool from the join kernel, with the stored rows as queries, and shares step 3.  Algorithmic bytes:
// ntotal * dpad * 2 per query chunk, plus 12 bytes per hit in the pool and 12 in the output.
#include "mma_common.cuh"

#include <climits>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>

namespace ivr {

__device__ __forceinline__ int64_t stored_hits(const unsigned long long* cursor, int64_t capacity) {
    const unsigned long long total = *cursor;
    return total > static_cast<unsigned long long>(capacity) ? 0 : static_cast<int64_t>(total);
}

__global__ void range_histogram_kernel(const uint32_t* __restrict__ qidx, const unsigned long long* __restrict__ cursor,
                                       int64_t capacity, unsigned long long* __restrict__ counts) {
    const int64_t n = stored_hits(cursor, capacity);
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x)
        atomicAdd(counts + qidx[i], 1ull);
}

__global__ void range_scatter_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ qidx,
                                     const unsigned long long* __restrict__ cursor, int64_t capacity,
                                     const int64_t* __restrict__ lims, unsigned long long* __restrict__ fill,
                                     uint64_t* __restrict__ out) {
    const int64_t n = stored_hits(cursor, capacity);
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const uint32_t q = qidx[i];
        out[lims[q] + static_cast<int64_t>(atomicAdd(fill + q, 1ull))] = keys[i];
    }
}

// D = score * q_scale[q], I = row + id_offset; the query of position i is found by bisection of lims
__global__ void range_unpack_kernel(const uint64_t* __restrict__ keys, const unsigned long long* __restrict__ cursor,
                                    int64_t capacity, const int64_t* __restrict__ lims, int64_t nq,
                                    const float* __restrict__ q_scale, int64_t id_offset, float* __restrict__ D,
                                    int64_t* __restrict__ I) {
    const int64_t n = stored_hits(cursor, capacity);
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        int64_t lo = 0, hi = nq - 1;                     // the q with lims[q] <= i < lims[q + 1]
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) >> 1;
            if (lims[mid] <= i) lo = mid; else hi = mid - 1;
        }
        const uint64_t key = keys[i];
        D[i] = key_score(key) * q_scale[lo];
        I[i] = static_cast<int64_t>(key_row(key)) + id_offset;
    }
}

// keys[i] = make_key(score * q_scale[q], row + id_offset), the exchange key of ivr_index_search_keys_device.  q_scale
// is a power of two, so the rescaled keys keep the segmented sort's order (score descending, then lower row).
__global__ void range_pack_keys_kernel(const uint64_t* __restrict__ sorted,
                                       const unsigned long long* __restrict__ cursor, int64_t capacity,
                                       const int64_t* __restrict__ lims, int64_t nq, const float* __restrict__ q_scale,
                                       int64_t id_offset, uint64_t* __restrict__ keys) {
    const int64_t n = stored_hits(cursor, capacity);
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        int64_t lo = 0, hi = nq - 1;
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) >> 1;
            if (lims[mid] <= i) lo = mid; else hi = mid - 1;
        }
        const uint64_t key = sorted[i];
        keys[i] = make_key(key_score(key) * q_scale[lo], key_row(key) + static_cast<uint32_t>(id_offset));
    }
}

// The hit pool and its grouping, shared by range search and the self-join.  `carve` holds the caller's own workspace
// parts; the pool's follow.  score(ws, cursor, keys, qidx) queues the launches that fill the pool of `capacity` (key,
// segment) entries; the segments [0, nq) are then grouped on the device: histogram, scan into lims, scatter, segmented
// sort descending (score descending, then lower row); finish(ws, sorted, cursor, grid, threads) queues the last step,
// which writes the caller's output.  lims[nq] ends as the exact total.
template <class Score, class Finish>
static int range_pool_sorted(ivr_index* idx, Carve carve, int64_t nq, int64_t capacity, int64_t* lims, cudaStream_t st,
                             Score&& score, Finish&& finish) {
    const int items = static_cast<int>(capacity);        // the caller checked capacity <= INT_MAX
    size_t scan_bytes = 0, sort_bytes = 0;
    IVR_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, static_cast<const int64_t*>(nullptr),
                                           static_cast<int64_t*>(nullptr), static_cast<int>(nq + 1), st));
    IVR_CUDA(cub::DeviceSegmentedSort::SortKeysDescending(nullptr, sort_bytes, static_cast<const uint64_t*>(nullptr),
                                                          static_cast<uint64_t*>(nullptr), items, static_cast<int>(nq),
                                                          static_cast<const int64_t*>(nullptr),
                                                          static_cast<const int64_t*>(nullptr), st));
    const size_t zero_bytes = (1 + 2 * static_cast<size_t>(nq) + 1) * 8;   // cursor, counts [nq + 1], fill [nq]
    const size_t o_z   = carve(zero_bytes);
    const size_t o_k   = carve(static_cast<size_t>(capacity) * 8);
    const size_t o_qi  = carve(static_cast<size_t>(capacity) * 4);
    const size_t o_seg = carve(static_cast<size_t>(capacity) * 8);
    const size_t o_srt = carve(static_cast<size_t>(capacity) * 8);
    const size_t o_tmp = carve(std::max(scan_bytes, sort_bytes));
    IVR_TRY(ensure_ws(idx, carve.size));
    char* ws = static_cast<char*>(idx->ws);
    unsigned long long* cursor = reinterpret_cast<unsigned long long*>(ws + o_z);
    unsigned long long* counts = cursor + 1;
    unsigned long long* fill = counts + nq + 1;
    uint64_t* keys = reinterpret_cast<uint64_t*>(ws + o_k);
    uint32_t* qidx = reinterpret_cast<uint32_t*>(ws + o_qi);
    uint64_t* seg = reinterpret_cast<uint64_t*>(ws + o_seg);
    uint64_t* sorted = reinterpret_cast<uint64_t*>(ws + o_srt);
    void* tmp = ws + o_tmp;

    IVR_CUDA(cudaMemsetAsync(cursor, 0, zero_bytes, st));
    IVR_TRY(score(ws, cursor, keys, qidx));
    const int grid = idx->sm_count * 4, threads = 256;
    range_histogram_kernel<<<grid, threads, 0, st>>>(qidx, cursor, capacity, counts);
    IVR_CUDA(cudaGetLastError());
    IVR_CUDA(cub::DeviceScan::ExclusiveSum(tmp, scan_bytes, reinterpret_cast<const int64_t*>(counts), lims,
                                           static_cast<int>(nq + 1), st));
    range_scatter_kernel<<<grid, threads, 0, st>>>(keys, qidx, cursor, capacity, lims, fill, seg);
    IVR_CUDA(cudaGetLastError());
    if (items > 0)
        IVR_CUDA(cub::DeviceSegmentedSort::SortKeysDescending(tmp, sort_bytes, seg, sorted, items, static_cast<int>(nq),
                                                              lims, lims + 1, st));
    IVR_TRY(finish(static_cast<const char*>(ws), static_cast<const uint64_t*>(sorted),
                   static_cast<const unsigned long long*>(cursor), grid, threads));
    // lims[nq] = the true total: equal to the scan's when the pool held every hit, the size to retry with otherwise
    IVR_CUDA(cudaMemcpyAsync(lims + nq, cursor, sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    return IVR_OK;
}

// The body shared by both range entry points: score every query chunk into the pool, group and sort it into lims /
// the sorted pool, then finish(sorted, cursor, q_scale, grid, threads) queues the last step, which writes the
// caller's output.
// With a cut of a selection, only the rows it selects are scored, and a cut without a tile scores nothing.
template <class Finish>
static int range_search_sorted(ivr_index* idx, const float* q_dev, int64_t nq, float radius, int64_t capacity,
                               int64_t* lims, cudaStream_t st, Finish&& finish, const SelCut* cut = nullptr) {
    if (idx->ntotal == 0 || (cut && cut->n_tiles == 0)) {
        IVR_CUDA(cudaMemsetAsync(lims, 0, static_cast<size_t>(nq + 1) * sizeof(int64_t), st));
        return IVR_OK;
    }
    const int chunk = small_range_chunk(idx);
    const int64_t n_chunks = (nq + chunk - 1) / chunk;
    Carve carve;
    const size_t o_q   = carve(static_cast<size_t>(chunk) * idx->dpad * 2);
    const size_t o_sc  = carve(static_cast<size_t>(n_chunks) * chunk * 4);
    const size_t o_tg  = carve(static_cast<size_t>(chunk) * 4);
    return range_pool_sorted(idx, carve, nq, capacity, lims, st,
                             [&](char* ws, unsigned long long* cursor, uint64_t* keys, uint32_t* qidx) {
        __half* q_h = reinterpret_cast<__half*>(ws + o_q);
        float* q_scale = reinterpret_cast<float*>(ws + o_sc);
        uint32_t* tau_g = reinterpret_cast<uint32_t*>(ws + o_tg);
        for (int64_t c = 0; c < n_chunks; ++c) {
            const int64_t q0 = c * chunk, m = std::min<int64_t>(chunk, nq - q0);
            IVR_TRY(launch_queries_to_f16(q_dev + q0 * idx->dim, q_h, q_scale + q0, tau_g, m, (m + 15) / 16 * 16,
                                          idx->dim, idx->dpad, st));
            IVR_TRY(search_mma_small_range(idx, q_h, q_scale + q0, m, q0, radius, cursor, keys, qidx, capacity, st,
                                           cut));
        }
        return IVR_OK;
    }, [&](const char* ws, const uint64_t* sorted, const unsigned long long* cursor, int grid, int threads) {
        return finish(sorted, cursor, reinterpret_cast<const float*>(ws + o_sc), grid, threads);
    });
}

// range search with the hits unpacked to D / I (cut == nullptr: every row)
static int range_search_unpacked(ivr_index* idx, const SelCut* cut, const float* q_dev, int64_t nq, float radius,
                                 int64_t capacity, int64_t* lims, float* D, int64_t* I, int64_t id_offset,
                                 cudaStream_t st) {
    return range_search_sorted(idx, q_dev, nq, radius, capacity, lims, st,
                               [&](const uint64_t* sorted, const unsigned long long* cursor, const float* q_scale,
                                   int grid, int threads) {
        range_unpack_kernel<<<grid, threads, 0, st>>>(sorted, cursor, capacity, lims, nq, q_scale, id_offset, D, I);
        IVR_CUDA(cudaGetLastError());
        return IVR_OK;
    }, cut);
}

// range search with the hits left as exchange keys (cut == nullptr: every row)
static int range_search_packed(ivr_index* idx, const SelCut* cut, const float* q_dev, int64_t nq, float radius,
                               int64_t capacity, int64_t* lims, uint64_t* keys, int64_t id_offset, cudaStream_t st) {
    return range_search_sorted(idx, q_dev, nq, radius, capacity, lims, st,
                               [&](const uint64_t* sorted, const unsigned long long* cursor, const float* q_scale,
                                   int grid, int threads) {
        range_pack_keys_kernel<<<grid, threads, 0, st>>>(sorted, cursor, capacity, lims, nq, q_scale, id_offset,
                                                         keys);
        IVR_CUDA(cudaGetLastError());
        return IVR_OK;
    }, cut);
}

int range_search_selected_device(ivr_index* idx, const SelCut& cut, const float* q_dev, int64_t nq, float radius,
                                 int64_t capacity, int64_t* lims, float* D, int64_t* I, int64_t id_offset,
                                 cudaStream_t st) {
    return range_search_unpacked(idx, &cut, q_dev, nq, radius, capacity, lims, D, I, id_offset, st);
}

int range_search_device(ivr_index* idx, const float* q_dev, int64_t nq, float radius, int64_t capacity,
                        int64_t* lims, float* D, int64_t* I, int64_t id_offset, cudaStream_t st) {
    return range_search_unpacked(idx, nullptr, q_dev, nq, radius, capacity, lims, D, I, id_offset, st);
}

int range_search_selected_keys_device(ivr_index* idx, const SelCut& cut, const float* q_dev, int64_t nq, float radius,
                                      int64_t capacity, int64_t* lims, uint64_t* keys, int64_t id_offset,
                                      cudaStream_t st) {
    return range_search_packed(idx, &cut, q_dev, nq, radius, capacity, lims, keys, id_offset, st);
}

int range_search_keys_device(ivr_index* idx, const float* q_dev, int64_t nq, float radius, int64_t capacity,
                             int64_t* lims, uint64_t* keys, int64_t id_offset, cudaStream_t st) {
    return range_search_packed(idx, nullptr, q_dev, nq, radius, capacity, lims, keys, id_offset, st);
}

__global__ void range_fill_kernel(float* __restrict__ x, int64_t n, float v) {
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x)
        x[i] = v;
}

// The joins' pool over nseg segments: score(cursor, keys, qidx) fills it, the grouping is range search's, and
// finish(sorted, cursor, ones, grid, threads) writes the output with scales of one (join scores are not rescaled).
template <class Score, class Finish>
static int join_pool_sorted(ivr_index* idx, int64_t nseg, int64_t capacity, int64_t* lims, cudaStream_t st,
                            Score&& score, Finish&& finish) {
    Carve carve;
    const size_t o_one = carve(static_cast<size_t>(nseg) * 4);
    return range_pool_sorted(idx, carve, nseg, capacity, lims, st,
                             [&](char*, unsigned long long* cursor, uint64_t* keys, uint32_t* qidx) {
        return score(cursor, keys, qidx);
    }, [&](const char* ws, const uint64_t* sorted, const unsigned long long* cursor, int grid, int threads) {
        float* ones = reinterpret_cast<float*>(const_cast<char*>(ws) + o_one);
        range_fill_kernel<<<grid, threads, 0, st>>>(ones, nseg, 1.0f);
        IVR_CUDA(cudaGetLastError());
        return finish(sorted, cursor, static_cast<const float*>(ones), grid, threads);
    });
}

// lims, D, I = range_self_join(radius): the join kernel (search_mma_small.cu) puts both (i, j) and (j, i) of every
// pair into the pool, segmented by the first row; the grouping is range search's, and the unpack's scales are ones.
int range_self_join_device(ivr_index* idx, float radius, int64_t capacity, int64_t* lims, float* D, int64_t* I,
                           int64_t id_offset, cudaStream_t st) {
    const int64_t n = idx->ntotal;
    if (n == 0) {
        IVR_CUDA(cudaMemsetAsync(lims, 0, sizeof(int64_t), st));
        return IVR_OK;
    }
    return join_pool_sorted(idx, n, capacity, lims, st, [&](unsigned long long* cursor, uint64_t* keys, uint32_t* qidx) {
        return search_mma_small_join(idx, radius, cursor, keys, qidx, capacity, st);
    }, [&](const uint64_t* sorted, const unsigned long long* cursor, const float* ones, int grid, int threads) {
        range_unpack_kernel<<<grid, threads, 0, st>>>(sorted, cursor, capacity, lims, n, ones, id_offset, D, I);
        IVR_CUDA(cudaGetLastError());
        return IVR_OK;
    });
}

// The self-join with its hits left as exchange keys (ShardedFlatIP.range_self_join: a rank's own window).
int range_self_join_keys_device(ivr_index* idx, float radius, int64_t capacity, int64_t* lims, uint64_t* keys,
                                int64_t id_offset, cudaStream_t st) {
    const int64_t n = idx->ntotal;
    if (n == 0) {
        IVR_CUDA(cudaMemsetAsync(lims, 0, sizeof(int64_t), st));
        return IVR_OK;
    }
    return join_pool_sorted(idx, n, capacity, lims, st, [&](unsigned long long* cursor, uint64_t* pool, uint32_t* qidx) {
        return search_mma_small_join(idx, radius, cursor, pool, qidx, capacity, st);
    }, [&](const uint64_t* sorted, const unsigned long long* cursor, const float* ones, int grid, int threads) {
        range_pack_keys_kernel<<<grid, threads, 0, st>>>(sorted, cursor, capacity, lims, n, ones, id_offset, keys);
        IVR_CUDA(cudaGetLastError());
        return IVR_OK;
    });
}

// The current rows against `other`: the cross-join kernel writes keys of global ids already, so the pack adds no
// offset.  Segments [0, n) are the current rows, [n, n + n_other) the other rows; an empty side scores nothing.
int range_cross_join_keys_device(ivr_index* idx, const __half* other, int64_t n_other, bool other_is_lower,
                                 uint32_t self_id0, uint32_t other_id0, float radius, int64_t capacity, int64_t* lims,
                                 uint64_t* keys, cudaStream_t st) {
    const int64_t n = idx->ntotal, nseg = n + n_other;
    if (n == 0 || n_other == 0) {
        IVR_CUDA(cudaMemsetAsync(lims, 0, static_cast<size_t>(nseg + 1) * sizeof(int64_t), st));
        return IVR_OK;
    }
    return join_pool_sorted(idx, nseg, capacity, lims, st,
                            [&](unsigned long long* cursor, uint64_t* pool, uint32_t* qidx) {
        return search_mma_small_cross_join(idx, other, n_other, other_is_lower, self_id0, other_id0, radius, cursor,
                                           pool, qidx, capacity, st);
    }, [&](const uint64_t* sorted, const unsigned long long* cursor, const float* ones, int grid, int threads) {
        range_pack_keys_kernel<<<grid, threads, 0, st>>>(sorted, cursor, capacity, lims, nseg, ones, 0, keys);
        IVR_CUDA(cudaGetLastError());
        return IVR_OK;
    });
}

// ---- merge of per-rank range runs (ShardedFlatIP.range_search) ----

// lims[q] = sum over parts of lims_parts[p][q]
__global__ void range_merge_lims_kernel(const int64_t* __restrict__ lims_parts, int n_parts, int64_t nq,
                                        int64_t* __restrict__ lims) {
    for (int64_t q = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; q <= nq;
         q += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        int64_t s = 0;
        for (int p = 0; p < n_parts; ++p) s += lims_parts[p * (nq + 1) + q];
        lims[q] = s;
    }
}

// One thread per input hit (p, j).  Its query q comes from bisecting lims_parts[p]; its output slot is
//   sum_s lims_parts[s][q]  +  (j - lims_parts[p][q])  +  sum_{s != p} |{keys of run (s, q) that come before it}|,
// the count found by binary search in each other (descending) run: keys greater than it, and in a lower part also
// keys equal to it.  This is the rank of (key, part, position) in one total order, so the slots are a permutation of
// query q's output range, also when two parts hold the same key.  Every slot stays inside [lims[q], lims[q + 1]).
__global__ void range_merge_keys_kernel(const uint64_t* __restrict__ keys_parts, int64_t part_stride,
                                        const int64_t* __restrict__ lims_parts, int n_parts, int64_t nq,
                                        float* __restrict__ D, int64_t* __restrict__ I) {
    const int64_t n = static_cast<int64_t>(n_parts) * part_stride;
    for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < n;
         t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int p = static_cast<int>(t / part_stride);
        const int64_t j = t - p * part_stride;
        const int64_t* lp = lims_parts + p * (nq + 1);
        if (j >= lp[nq]) continue;
        int64_t lo = 0, hi = nq - 1;                     // the q with lp[q] <= j < lp[q + 1]
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) >> 1;
            if (lp[mid] <= j) lo = mid; else hi = mid - 1;
        }
        const int64_t q = lo;
        const uint64_t key = keys_parts[t];
        int64_t slot = j - lp[q];
        for (int s = 0; s < n_parts; ++s) {
            const int64_t* ls = lims_parts + s * (nq + 1);
            const int64_t b = ls[q], e = ls[q + 1];
            slot += b;
            if (s == p) continue;
            const uint64_t* run = keys_parts + s * part_stride;
            int64_t a = b, z = e;                        // first position in [b, e) that comes after `key`
            if (s < p) { while (a < z) { const int64_t m = (a + z) >> 1; if (run[m] >= key) a = m + 1; else z = m; } }
            else       { while (a < z) { const int64_t m = (a + z) >> 1; if (run[m] > key) a = m + 1; else z = m; } }
            slot += a - b;
        }
        D[slot] = key_score(key);
        I[slot] = static_cast<int64_t>(key_row(key));
    }
}

int range_merge_keys_device(const uint64_t* keys_parts, int64_t part_stride, const int64_t* lims_parts, int n_parts,
                            int64_t nq, int64_t* lims, float* D, int64_t* I, cudaStream_t st) {
    const int threads = 256;
    const int64_t grid_cap = 2048;                       // grid-stride beyond that: enough blocks to fill 148 SMs
    const int g_lims = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((nq + threads) / threads, grid_cap)));
    range_merge_lims_kernel<<<g_lims, threads, 0, st>>>(lims_parts, n_parts, nq, lims);
    IVR_CUDA(cudaGetLastError());
    const int64_t n = static_cast<int64_t>(n_parts) * part_stride;
    if (n == 0) return IVR_OK;
    const int g = static_cast<int>(std::min<int64_t>((n + threads - 1) / threads, grid_cap));
    range_merge_keys_kernel<<<g, threads, 0, st>>>(keys_parts, part_stride, lims_parts, n_parts, nq, D, I);
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

}  // namespace ivr

// selection.cu -- device row selections for filtered search (ivr_selection_create).
//
// A selection is a packed bitmap over stored rows (bit i & 31 of word i >> 5 = row i) plus the ascending list of the
// 128-row tiles that hold at least one selected row.  A tile is four bitmap words -- the 32 rows each epilogue warp
// of the small-batch kernel drains -- so the list is one OR per tile and a compaction.  Both are built once per
// selection and read by every filtered search: the producer warp streams tiles[j], the epilogue warps AND their
// word into the row-validity test (search_mma_small.cu).  100 M rows: 12.5 MB of bitmap, at most 3 MB of tile list.
// The host keeps a copy of both, so that a search can cut a window's tiles out of the list without touching the device
// (selection_cut): the sharded index searches a different window of the same selection whenever its boundaries move.
#include "index.cuh"

#include <cub/device/device_select.cuh>
#include <new>

namespace ivr {

// flags[t] = tile t holds a selected row; the bits of rows at or past n_rows are cleared on the way
__global__ void selection_flags_kernel(uint32_t* __restrict__ words, int64_t n_rows, int64_t n_tiles,
                                       uint8_t* __restrict__ flags) {
    for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < n_tiles;
         t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        uint32_t any = 0;
        for (int i = 0; i < 4; ++i) {
            const int64_t w = t * 4 + i, row0 = w * 32;
            uint32_t word = words[w];
            if (row0 + 32 > n_rows) {
                word &= row0 >= n_rows ? 0u : (1u << (n_rows - row0)) - 1u;
                words[w] = word;
            }
            any |= word;
        }
        flags[t] = any != 0;
    }
}

__global__ void selection_iota_kernel(uint32_t* __restrict__ ids, int64_t n) {
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x)
        ids[i] = static_cast<uint32_t>(i);
}

int selection_destroy(ivr_selection* sel) {
    if (!sel) return IVR_OK;
    cudaSetDevice(sel->device);
    cudaFree(sel->words);
    cudaFree(sel->tiles);
    delete sel;
    return IVR_OK;
}

int selection_create(int device, const uint32_t* words_host, int64_t n_rows, ivr_selection** out) {
    ivr_selection* sel = new (std::nothrow) ivr_selection;
    if (!sel) { set_error("selection_create: out of host memory"); return IVR_ENOMEM; }
    sel->device = device;
    sel->n_rows = n_rows;
    const int64_t n_tiles = (n_rows + 127) / 128, n_words = (n_rows + 31) / 32;
    sel->words_host.resize(static_cast<size_t>(n_words));
    for (int64_t w = 0; w < n_words; ++w) {
        const int64_t left = n_rows - w * 32;
        const uint32_t word = left >= 32 ? words_host[w] : words_host[w] & ((1u << left) - 1u);
        sel->words_host[w] = word;
        sel->count += __builtin_popcount(word);
    }
    if (n_tiles == 0) { *out = sel; return IVR_OK; }

    cudaStream_t st = nullptr;
    uint8_t* flags = nullptr;
    uint32_t* ids = nullptr;
    int* n_sel = nullptr;
    void* tmp = nullptr;
    auto run = [&]() -> int {
        IVR_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        const size_t wb = static_cast<size_t>(n_tiles) * 16;
        if (cudaMalloc(&sel->words, wb) != cudaSuccess || cudaMalloc(&sel->tiles, n_tiles * 4) != cudaSuccess ||
            cudaMalloc(&flags, n_tiles) != cudaSuccess || cudaMalloc(&ids, n_tiles * 4) != cudaSuccess ||
            cudaMalloc(&n_sel, sizeof(int)) != cudaSuccess) {
            cudaGetLastError();
            set_error("selection_create: device allocation of %lld bytes failed", static_cast<long long>(wb * 2));
            return IVR_ENOMEM;
        }
        IVR_CUDA(cudaMemsetAsync(sel->words, 0, wb, st));
        IVR_CUDA(cudaMemcpyAsync(sel->words, words_host, static_cast<size_t>(n_words) * 4, cudaMemcpyHostToDevice, st));
        const int threads = 256;
        const int grid = static_cast<int>(std::min<int64_t>((n_tiles + threads - 1) / threads, 4096));
        selection_flags_kernel<<<grid, threads, 0, st>>>(sel->words, n_rows, n_tiles, flags);
        IVR_CUDA(cudaGetLastError());
        selection_iota_kernel<<<grid, threads, 0, st>>>(ids, n_tiles);
        IVR_CUDA(cudaGetLastError());
        size_t tmp_bytes = 0;
        const int n = static_cast<int>(n_tiles);                   // < 2^25: n_rows <= 2^32
        IVR_CUDA(cub::DeviceSelect::Flagged(nullptr, tmp_bytes, ids, flags, sel->tiles, n_sel, n, st));
        IVR_CUDA(cudaMalloc(&tmp, tmp_bytes));
        IVR_CUDA(cub::DeviceSelect::Flagged(tmp, tmp_bytes, ids, flags, sel->tiles, n_sel, n, st));
        int n_list = 0;
        IVR_CUDA(cudaMemcpyAsync(&n_list, n_sel, sizeof(int), cudaMemcpyDeviceToHost, st));
        IVR_CUDA(cudaStreamSynchronize(st));
        sel->tiles_host.resize(static_cast<size_t>(n_list));
        if (n_list)
            IVR_CUDA(cudaMemcpyAsync(sel->tiles_host.data(), sel->tiles, static_cast<size_t>(n_list) * 4,
                                     cudaMemcpyDeviceToHost, st));
        IVR_CUDA(cudaStreamSynchronize(st));
        return IVR_OK;
    };
    const int rc = run();
    cudaFree(flags); cudaFree(ids); cudaFree(n_sel); cudaFree(tmp);
    if (st) cudaStreamDestroy(st);
    if (rc != IVR_OK) { selection_destroy(sel); return rc; }
    *out = sel;
    return IVR_OK;
}

// position of the first tile id >= t in the selection's tile list
static int64_t tile_pos(const ivr_selection* sel, int64_t t) {
    return std::lower_bound(sel->tiles_host.begin(), sel->tiles_host.end(), static_cast<uint64_t>(t),
                            [](uint32_t v, uint64_t x) { return v < x; }) - sel->tiles_host.begin();
}

int64_t selection_tiles(const ivr_selection* sel, int64_t ntotal) { return tile_pos(sel, (ntotal + 127) / 128); }

SelCut selection_all(const ivr_selection* sel, int64_t ntotal) {
    return SelCut{sel->tiles, sel->words, selection_tiles(sel, ntotal), 0, ntotal};
}

// whether the host bitmap selects a row of [a, b)
static bool any_selected(const ivr_selection* sel, int64_t a, int64_t b) {
    b = std::min(b, sel->n_rows);
    for (int64_t r = a; r < b; ++r)
        if ((sel->words_host[r >> 5] >> (r & 31)) & 1u) return true;
    return false;
}

// The tiles from first / 128 to ceil(end / 128) by two binary searches; a partial first or last tile whose selected rows
// all lie outside the window is dropped, so an empty cut means "no selected row in the window".
SelCut selection_cut(const ivr_selection* sel, int64_t first, int64_t end) {
    int64_t lo = tile_pos(sel, first / 128), hi = tile_pos(sel, (end + 127) / 128);
    if (lo < hi && first % 128 != 0 && sel->tiles_host[lo] == first / 128 &&
        !any_selected(sel, first, std::min(end, (first / 128 + 1) * 128)))
        ++lo;
    if (lo < hi && end % 128 != 0 && sel->tiles_host[hi - 1] == end / 128 &&
        !any_selected(sel, std::max(first, end / 128 * 128), end))
        --hi;
    return SelCut{sel->tiles + lo, sel->words, hi - lo, first, end};
}

}  // namespace ivr

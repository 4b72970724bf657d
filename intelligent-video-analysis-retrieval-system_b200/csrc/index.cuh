// index.cuh -- the flat inner-product index handle (device-resident fp16 rows).
#pragma once

#include "common.cuh"

#include <vector>

namespace ivr {
// Event slots of the search timing (ivr_index_last_timing): interval i runs from ev[2i] to ev[2i + 1], so
// score_ms = scoring launches, merge_ms = the final merge, prep_ms = query preparation.
enum TimingMark { kScoreBegin = 0, kScoreEnd = 1, kMergeBegin = 2, kMergeEnd = 3, kPrepBegin = 4, kPrepEnd = 5 };
}  // namespace ivr

struct ivr_index {
    int      dim      = 0;        // logical dimension (as given by the caller)
    int      dpad     = 0;        // storage dimension: dim padded to a multiple of 64
    int      device   = 0;
    int      sm_count = 0;
    int64_t  ntotal   = 0;
    int64_t  capacity = 0;        // rows allocated
    __half* rows = nullptr;          // [capacity, dpad] row-major fp16, HBM

    // search window (ivr_index_set_window): searches score rows [win_first, win_first + win_count) only;
    // win_count < 0 = the whole index
    int64_t  win_first = 0, win_count = -1;

    cudaStream_t stream = nullptr;   // handle-owned stream for the host-pointer entry points

    // scratch, grown on demand (device)
    void*   ws      = nullptr;
    size_t  ws_bytes = 0;
    // device staging for the host-pointer search entry point (queries in, D/I out)
    void*   io       = nullptr;
    size_t  io_bytes = 0;
    // pinned host staging
    void*   pin      = nullptr;
    size_t  pin_bytes = 0;
    // counters / tickets of the one-launch select merge (topk_merge.cu): zeroed at creation, re-zeroed by the kernel itself
    int*    sel_state = nullptr;

    // TMA descriptor cache for the MMA path (opaque 128-byte CUtensorMap blobs)
    alignas(64) unsigned char tmap_rows[128];
    const void* tmap_rows_base = nullptr;
    int64_t     tmap_rows_n    = -1;
    int         tmap_rows_box  = 0;

    // recorded after every device-side add on its stream; searches on other streams wait on it
    cudaEvent_t rows_ready = nullptr;
    bool        rows_ready_set = false;

    // timing of the last device search
    bool        timing = false;
    cudaEvent_t ev[6]  = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // indexed by ivr::TimingMark
    bool        ev_valid[3] = {false, false, false};
    int         launches[3] = {0, 0, 0};
    int         last_path = 0;
    const char* last_kernel = "";
};

// A device row selection (ivr_selection_create, selection.cu): bit i & 31 of word i >> 5 selects stored row i.
struct ivr_selection {
    int       device = 0;
    int64_t   n_rows = 0;              // rows the bitmap covers; rows at or past n_rows are not selected
    int64_t   count  = 0;              // selected rows
    uint32_t* words  = nullptr;        // [4 * ceil(n_rows / 128)] device bitmap, zero from row n_rows on
    uint32_t* tiles  = nullptr;        // device, ascending: the 128-row tiles that hold a selected row
    std::vector<uint32_t> tiles_host;  // the same list, to cut it at an index's tile count or to a search window
    std::vector<uint32_t> words_host;  // the bitmap, to trim a window's partial first and last tiles
};

namespace ivr {

int  ensure_ws(ivr_index* idx, size_t bytes);
int  ensure_pin(ivr_index* idx, size_t bytes);
int  ensure_io(ivr_index* idx, size_t bytes);
int  ensure_capacity(ivr_index* idx, int64_t rows, cudaStream_t st, bool exact = false);

// Records timing mark m of the current search on st when `timed`.
inline void timing_mark(ivr_index* idx, bool timed, TimingMark m, cudaStream_t st) {
    if (timed) cudaEventRecord(idx->ev[m], st);
}

// Consecutive 256-byte-aligned parts of one buffer: carve(bytes) returns the next part's offset, `size` the total.
struct Carve {
    size_t size = 0;
    size_t operator()(size_t bytes) { const size_t o = size; size += (bytes + 255) / 256 * 256; return o; }
};

// search back-ends (search_stream.cu / search_mma.cu / topk_merge.cu)
int search_stream(ivr_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev,
                  int64_t* I_dev, int64_t id_offset, cudaStream_t st);
int search_mma(ivr_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev,
               int64_t* I_dev, int64_t id_offset, cudaStream_t st);
bool mma_supported(const ivr_index* idx, int64_t nq, int k);
bool mma_small_supported(const ivr_index* idx, int64_t nq, int k);   // small-batch kernel (search_mma_small.cu)
int  small_range_chunk(const ivr_index* idx);    // queries per range launch of that kernel; 0 = dimension too wide
// lims, D, I = range_search(q, radius) on the current rows (range_search.cu); capacity <= INT_MAX
int  range_search_device(ivr_index* idx, const float* q_dev, int64_t nq, float radius, int64_t capacity,
                         int64_t* lims, float* D, int64_t* I, int64_t id_offset, cudaStream_t st);
// the same search, hits left as exchange keys make_key(score, row + id_offset) in the order of D / I
int  range_search_keys_device(ivr_index* idx, const float* q_dev, int64_t nq, float radius, int64_t capacity,
                              int64_t* lims, uint64_t* keys, int64_t id_offset, cudaStream_t st);
// lims [ntotal + 1], D, I = every pair of distinct current rows with score > radius, by first row (range_search.cu)
int  range_self_join_device(ivr_index* idx, float radius, int64_t capacity, int64_t* lims, float* D, int64_t* I,
                            int64_t id_offset, cudaStream_t st);
// the same join, hits left as exchange keys make_key(score, row + id_offset) in the order of D / I
int  range_self_join_keys_device(ivr_index* idx, float radius, int64_t capacity, int64_t* lims, uint64_t* keys,
                                 int64_t id_offset, cudaStream_t st);
// every pair (current row i, other row j) with score > radius, as exchange keys of global ids: lims [n + n_other + 1]
// holds the current rows' segments, then the other rows'; current row i is global id self_id0 + i, other row j
// other_id0 + j (range_search.cu)
int  range_cross_join_keys_device(ivr_index* idx, const __half* other, int64_t n_other, bool other_is_lower,
                                  uint32_t self_id0, uint32_t other_id0, float radius, int64_t capacity, int64_t* lims,
                                  uint64_t* keys, cudaStream_t st);
// row selections (selection.cu): build the device bitmap and tile list of a new handle; the number of tiles of the
// list that lie below an index of ntotal rows
int  selection_create(int device, const uint32_t* words_host, int64_t n_rows, ivr_selection** out);
int  selection_destroy(ivr_selection* sel);
int64_t selection_tiles(const ivr_selection* sel, int64_t ntotal);
// What one filtered search streams and reports: the row tiles tiles[0 .. n_tiles) (a run of a selection's tile list)
// and, of their rows, the selected ones in [row_lo, row_hi).  Stored-row coordinates: a search window is not shifted
// to row 0 (RowWindow) but cut out here, because the selection's tile ids are stored tiles.
struct SelCut {
    const uint32_t* tiles;
    const uint32_t* words;
    int64_t n_tiles;
    int64_t row_lo, row_hi;
};
// every selected row below ntotal (the tiles of selection_tiles)
SelCut selection_all(const ivr_selection* sel, int64_t ntotal);
// the selected rows of the stored rows [first, end): the tiles that hold one, found on the host (no device sync)
SelCut selection_cut(const ivr_selection* sel, int64_t first, int64_t end);
// filtered top-k on the small-batch kernel (search_mma_small.cu) over `cut`, queries in chunks of small_sel_chunk();
// small_sel_chunk() == 0: the dimension or k does not fit.  D_dev == nullptr: packed keys into I_dev, as in search_mma
int  small_sel_chunk(const ivr_index* idx, int k);
int  search_mma_small_selected(ivr_index* idx, const SelCut& cut, const float* q_dev, int64_t nq, int k, float* D_dev,
                               int64_t* I_dev, int64_t id_offset, cudaStream_t st);
// range_search_device / range_search_keys_device over the selected rows of `cut` only (range_search.cu)
int  range_search_selected_device(ivr_index* idx, const SelCut& cut, const float* q_dev, int64_t nq, float radius,
                                  int64_t capacity, int64_t* lims, float* D, int64_t* I, int64_t id_offset,
                                  cudaStream_t st);
int  range_search_selected_keys_device(ivr_index* idx, const SelCut& cut, const float* q_dev, int64_t nq, float radius,
                                       int64_t capacity, int64_t* lims, uint64_t* keys, int64_t id_offset,
                                       cudaStream_t st);
// merge of per-part sorted range runs into lims / D / I (ivr_range_merge_keys_device); no scratch, two launches
int  range_merge_keys_device(const uint64_t* keys_parts, int64_t part_stride, const int64_t* lims_parts, int n_parts,
                             int64_t nq, int64_t* lims, float* D, int64_t* I, cudaStream_t st);

// Generic list merge.  For query q, list l lives at entries + l*list_stride + q*q_stride
// (64-bit keys) and holds counts[l*cnt_list_stride + q*cnt_q_stride] entries (or
// `fixed_count` entries when counts == nullptr).
struct MergeIn {
    const uint64_t* entries;
    const int*      counts;
    int64_t list_stride, q_stride;
    int64_t cnt_list_stride, cnt_q_stride;
    int     n_lists;
    int     fixed_count;
    int     raw;             // entries are raw {score bits, row} pairs (converted to keys on load)
    int     interleave;      // lists of 32 consecutive queries are interleaved: entry i of query q lives at
                             // l*list_stride + (q / 32) * q_stride * 32 + i * 32 + q % 32
    // DENSE mode (dense != nullptr; `entries` unused): list l of query q is the `dense_len` consecutive SCORES
    // dense[q * dense_q_stride + l * dense_len + i], i.e. rows l * dense_len + i (< dense_rows) of a materialised
    // score matrix; keys are formed on load.
    const float* dense;
    int64_t      dense_q_stride, dense_rows;
    int          dense_len;
};
// final stage: writes D/I ([nq,k], padded with -FLT_MAX / -1); ids = row + id_offset;
// scores are multiplied by q_scale[q] when q_scale != nullptr (power-of-two query scaling)
int merge_lists_final(const MergeIn& in, int64_t nq, int k, float* D_dev, int64_t* I_dev,
                      int64_t id_offset, uint64_t* tmp_entries, int* tmp_counts,
                      cudaStream_t st, int* n_launches, const float* q_scale = nullptr);
// one-launch merge for many short lists using the per-list maxima (topk_merge.cu); k <= kSelectMaxK
constexpr int kSelectMaxK    = 1024;
constexpr int kSelectPoolCap = 4096;
int merge_select_final(const MergeIn& in, const uint32_t* maxima, int64_t nq, int k, float* D_dev, int64_t* I_dev,
                       int64_t id_offset, uint64_t* pool, int* pool_cnt, int* ticket, int sm_count, cudaStream_t st,
                       int* n_launches, const float* q_scale = nullptr,
                       const uint32_t* group_max = nullptr, int n_groups = 0);   // [nq][n_groups]: bound searched in these
int merge_lists_keys(const MergeIn& in, int64_t nq, int k, uint64_t* out_keys, int* out_counts,
                     uint64_t* tmp_entries, int* tmp_counts, cudaStream_t st, int* n_launches);
size_t merge_tmp_entries(int n_lists, int64_t nq, int k);   // #keys of scratch the merge may need

}  // namespace ivr

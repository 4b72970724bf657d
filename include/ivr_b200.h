/*
 * ivr_b200.h -- C ABI of the B200-native retrieval hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b, level B2).  The reference
 * (DMDung2k3/Intelligent-Video-Analysis-Retrieval-System) is pure Python and
 * hands this arithmetic to third-party libraries; each entry point below names
 * the reference call it replaces.  The Python host in
 * intelligent-video-analysis-retrieval-system_b200/ binds these symbols with
 * ctypes (see INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / numpy types.
 *   - every function returns 0 (IVR_OK) or a negative IVR_E* code; a
 *     thread-local message is available from ivr_last_error().
 *   - "*_device" variants take DEVICE pointers on the handle's GPU and a
 *     cudaStream_t (as void*; NULL = the legacy default stream, exactly as in
 *     the CUDA runtime) and never block the host; the plain variants take HOST
 *     pointers, run on a stream owned by the handle, do the H2D/D2H copies
 *     themselves and return when the outputs are written.
 *   - there is NO CPU fallback: without a CUDA device every compute call
 *     fails with IVR_ENODEVICE.
 *   - a handle is not re-entrant (the reference serialises searches on an
 *     RLock: core.py:873, unified_index.py:92).
 */
#ifndef IVR_B200_H
#define IVR_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define IVR_API __attribute__((visibility("default")))
#else
#define IVR_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define IVR_OK          0
#define IVR_EINVAL     -1   /* bad argument (dimension mismatch, k <= 0, null pointer ...) */
#define IVR_ENODEVICE  -2   /* no usable CUDA device / wrong architecture                 */
#define IVR_ECUDA      -3   /* a CUDA runtime or driver call failed                        */
#define IVR_ENOMEM     -4   /* device or pinned-host allocation failed                     */
#define IVR_EUNSUPPORTED -5 /* argument outside the supported range (e.g. k > IVR_MAX_K)   */

#define IVR_MAX_K       2048  /* reference caps SearchOptions.limit at 1000 (system.py:83-92) */
#define IVR_MAX_WINDOW  32    /* dedup look-back window (reference default 5, config B uses 8) */

/* search path selector for ivr_index_search*(): */
#define IVR_PATH_AUTO    0
#define IVR_PATH_STREAM  1    /* K3: SIMT streaming, <= 4 queries per pass, HBM-bound (auto: nq == 1) */
#define IVR_PATH_MMA     2    /* K1+K2: tcgen05/TMEM batched GEMM with fused top-k epilogue   */

typedef struct ivr_index ivr_index;

/* ---- misc -------------------------------------------------------------- */
IVR_API const char* ivr_last_error(void);
IVR_API int         ivr_version(void);
IVR_API int         ivr_device_count(int* count);
/* name / SM count / total bytes of a device (any pointer may be NULL) */
IVR_API int         ivr_device_info(int device, char* name, size_t name_len, int* sm_count,
                            int* cc_major, int* cc_minor, size_t* total_bytes);

/* ---- flat inner-product index ------------------------------------------
 * Replaces faiss.IndexFlatIP(dim) + .add + .ntotal + .reset
 *   (unified_index.py:1767, 1779; core.py:1208, 827, 843, 268).
 * Rows are stored row-major in HBM as fp16 (dim padded to a multiple of 64;
 * values are saturated to +-65504 -- the reference only adds L2-normalised rows);
 * ids are the insertion order 0..ntotal-1.
 */
IVR_API int     ivr_index_create(int dim, int device, ivr_index** out);
IVR_API int     ivr_index_destroy(ivr_index* idx);
IVR_API int     ivr_index_reserve(ivr_index* idx, int64_t n_rows);           /* pre-size, avoids regrowth */
IVR_API int     ivr_index_add(ivr_index* idx, const float* x_host, int64_t n);
IVR_API int     ivr_index_add_device(ivr_index* idx, const float* x_dev, int64_t n, void* stream);
/* Replaces index.reconstruct_n(first, n) -- what faiss.write_index / serialize_index store for a flat index
 * (unified_index.py:1811; core.py:987): rows [first, first + n) as float32 [n, dim] (HOST pointer).  The values
 * are the stored fp16 rows widened exactly, i.e. the added rows after one rounding to fp16. */
IVR_API int     ivr_index_reconstruct(ivr_index* idx, int64_t first, int64_t n, float* x_host);
IVR_API int     ivr_index_reset(ivr_index* idx);
IVR_API int64_t ivr_index_ntotal(const ivr_index* idx);
IVR_API int     ivr_index_dim(const ivr_index* idx);
IVR_API int     ivr_index_device(const ivr_index* idx);

/* Replaces D, I = index.search(x, k)  (unified_index.py:503; core.py:891; system.py:1330).
 *   q      float32 [nq, dim] row-major
 *   D      float32 [nq, k]   inner products, descending
 *   I      int64   [nq, k]   row ids + id_offset; -1 (score -FLT_MAX) where k > ntotal
 * id_offset lets a row shard report global ids (multi-GPU row sharding).
 */
IVR_API int ivr_index_search(ivr_index* idx, const float* q_host, int64_t nq, int k,
                     float* D_host, int64_t* I_host, int path);
IVR_API int ivr_index_search_device(ivr_index* idx, const float* q_dev, int64_t nq, int k,
                            float* D_dev, int64_t* I_dev, int64_t id_offset, int path,
                            void* stream);

/* Same search, result left as PACKED candidate keys for the cross-shard exchange (8 bytes per hit instead of
 * 12): keys uint64 [nq, k] (device), key = order_preserving(float32 score) << 32 | ~(uint32)(row + id_offset),
 * unsigned descending order = score descending then lower id, key 0 = padding (k > ntotal).  Global row ids
 * must stay below 2^32 (id_offset + ntotal <= 2^32), else IVR_EUNSUPPORTED.  Merged by
 * ivr_topk_merge_keys_device after the exchange (ivr_exchange_* below, or one all-gather; semantic precedent:
 * system.py:1721-1746). */
IVR_API int ivr_index_search_keys_device(ivr_index* idx, const float* q_dev, int64_t nq, int k,
                                 uint64_t* keys_dev, int64_t id_offset, int path, void* stream);

/* Replaces lims, D, I = index.range_search(x, radius) of faiss.IndexFlatIP (not called by the reference): every
 * stored row whose inner product with the query is strictly greater than `radius`.
 *   lims   int64   [nq + 1]  the hits of query i are D[lims[i] : lims[i+1]], I[lims[i] : lims[i+1]]
 *   D      float32 [capacity] scores, descending within a query (ties -> lower id)
 *   I      int64   [capacity] row ids + id_offset
 * lims always receives nq + 1 entries.  When lims[nq] > capacity only lims[nq] (the exact total) is meaningful and
 * D / I are untouched: retry with capacity >= lims[nq] (the max_hits convention of ivr_sequence_similarity).
 * Scores, ids and the search window are those of ivr_index_search.  A NaN radius is IVR_EINVAL; capacity above
 * 2^31-1, padded dim above 4096 and indexes of 2^32 rows or more are IVR_EUNSUPPORTED.  The device variant never
 * blocks the host; its scratch grows the handle's workspace by about 28 bytes per capacity entry.  The host variant
 * stages through the handle's pinned buffer. */
IVR_API int ivr_index_range_search(ivr_index* idx, const float* q_host, int64_t nq, float radius, int64_t capacity,
                                   int64_t* lims_host, float* D_host, int64_t* I_host);
IVR_API int ivr_index_range_search_device(ivr_index* idx, const float* q_dev, int64_t nq, float radius,
                                          int64_t capacity, int64_t* lims_dev, float* D_dev, int64_t* I_dev,
                                          int64_t id_offset, void* stream);
/* The same range search, hits left as PACKED exchange keys (the format of ivr_index_search_keys_device):
 *   keys   uint64  [capacity] make_key(score, row + id_offset); query i's hits are keys[lims[i] : lims[i+1]], in the
 *                             order of D / I above (score descending, then lower id), so unsigned key descending
 * Same contract as ivr_index_range_search_device (capacity, the exact total in lims[nq], the search window, the
 * argument checks before any device call); in addition id_offset + ntotal > 2^32 is IVR_EUNSUPPORTED.  The per-rank
 * step of ShardedFlatIP.range_search: the runs of all ranks are merged by ivr_range_merge_keys_device. */
IVR_API int ivr_index_range_search_keys_device(ivr_index* idx, const float* q_dev, int64_t nq, float radius,
                                               int64_t capacity, int64_t* lims_dev, uint64_t* keys_dev,
                                               int64_t id_offset, void* stream);

/* Exact range self-join: every pair of distinct stored rows whose inner product is strictly greater than `radius`.
 * No reference call does this (the reference compares frames only within one scene or one folder); it finds the
 * same footage across videos: a shared intro, advert or news segment, or a re-upload.  The rows joined are those of
 * the search window (ivr_index_set_window), or all rows; call their count n.
 *   lims   int64   [n + 1]    row i's hits (i = position in the window) are D[lims[i] : lims[i+1]], I[...]
 *   D      float32 [capacity] scores, descending within a row (ties -> lower id)
 *   I      int64   [capacity] stored row ids (window first + position)
 * Row i's hits are the rows j != i with score(i, j) > radius, score = the fp32 tensor-core inner product of the two
 * stored fp16 rows (no query scaling).  Each pair is scored once, so the result is symmetric with equal score bits
 * both ways.  A row holding a NaN is never a hit and has no hits.  Apart from the diagonal, the result equals
 * ivr_index_range_search over the window's reconstructed rows wherever the two give the same fp32 score.  The capacity
 * convention is that of ivr_index_range_search: when lims[n] > capacity only lims[n] (the exact total) is meaningful
 * and D / I are untouched.  Checks, before any device call and in this order: a NaN radius, a negative capacity, a
 * NULL index or lims, or NULL D / I with capacity > 0 are IVR_EINVAL; capacity above 2^31-1, padded dim above 4096,
 * an index of 2^32 rows or more and a window of 2^31-1 rows or more are IVR_EUNSUPPORTED.  A window reaching beyond
 * the rows is IVR_EINVAL, and so many rows that the join needs more than 2^31-1 work units (about 50 M at 512 dims)
 * IVR_EUNSUPPORTED, when the call runs.  The device variant never blocks the host; its scratch grows the handle's
 * workspace by about 28 bytes per capacity entry and 36 bytes per row.  The host variant stages through the
 * handle's pinned buffer. */
IVR_API int ivr_index_range_self_join(ivr_index* idx, float radius, int64_t capacity, int64_t* lims_host,
                                      float* D_host, int64_t* I_host);
IVR_API int ivr_index_range_self_join_device(ivr_index* idx, float radius, int64_t capacity, int64_t* lims_dev,
                                             float* D_dev, int64_t* I_dev, void* stream);

/* ---- the pieces of a self-join across row shards (ShardedFlatIP.range_self_join) ------------------------------
 * The stored fp16 rows [first, first + n) (all stored rows, whatever the search window) copied to dst, dpad halves
 * per row (dpad = ivr_index_dpad: dim padded to a multiple of 64), with cudaMemcpyAsync on `stream`.  A NULL index,
 * NULL dst with n > 0, first < 0, n < 0 or a range past ntotal are IVR_EINVAL. */
IVR_API int ivr_index_dpad(const ivr_index* idx);
IVR_API int ivr_index_rows_f16_device(ivr_index* idx, int64_t first, int64_t n, void* dst, void* stream);
/* ivr_index_range_self_join_device with the hits left as PACKED exchange keys (the format of
 * ivr_index_search_keys_device): keys[lims[i] : lims[i+1]] = make_key(score, partner stored row + id_offset), in the
 * order of D / I.  Same contract and checks as ivr_index_range_self_join_device; in addition id_offset < 0 or
 * id_offset + ntotal > 2^32 is IVR_EUNSUPPORTED. */
IVR_API int ivr_index_range_self_join_keys_device(ivr_index* idx, float radius, int64_t capacity, int64_t* lims_dev,
                                                  uint64_t* keys_dev, int64_t id_offset, void* stream);
/* The rows of the search window (n_self of them; all stored rows without one) against n_other other rows: every
 * pair (window row i, other row j) whose inner product is strictly greater than `radius`, each pair scored once.
 *   other_rows      fp16 [n_other, dpad] on the index's device, global ids other_first_id + j
 *   other_is_lower  nonzero when the other rows' global ids are below the window's; that set is the streamed operand,
 *                   as the lower row i of a pair is in ivr_index_range_self_join, so a pair scores the same bits
 *   lims  int64  [n_self + n_other + 1]  window row i's hits are keys[lims[i] : lims[i+1]], other row j's are
 *                                        keys[lims[n_self + j] : lims[n_self + j + 1]]
 *   keys  uint64 [capacity]  make_key(score, global id of the partner), descending within a row; a window row's
 *                            global id is its stored row + id_offset
 * The capacity convention is that of ivr_index_range_search.  Checks, before any device call and in this order: a
 * NaN radius, a negative capacity or n_other, a NULL index, lims, keys with capacity > 0, or other_rows with
 * n_other > 0 are IVR_EINVAL; capacity above 2^31-1, padded dim above 4096, n_self + n_other of 2^31-1 or more, and a
 * global id reaching 2^32 (id_offset < 0, id_offset + ntotal > 2^32, other_first_id < 0 or other_first_id + n_other >
 * 2^32) are IVR_EUNSUPPORTED.  More than 2^31-1 work units run as several launches.  Never blocks the host. */
IVR_API int ivr_index_range_cross_join_keys_device(ivr_index* idx, const void* other_rows, int64_t n_other,
                                                   int64_t other_first_id, int other_is_lower, float radius,
                                                   int64_t capacity, int64_t* lims_dev, uint64_t* keys_dev,
                                                   int64_t id_offset, void* stream);

/* ---- filtered search: a device row selection -----------------------------------------------------------------
 * Replaces SearchParameters(sel=IDSelector...) on faiss.IndexFlatIP.search / range_search (the reference can only
 * post-filter the global top-k: unified_index.py:185-238).  A selection is built once from a packed host bitmap --
 * bit i & 31 of words[i >> 5] selects stored row i, for i < n_rows; rows at or past n_rows are not selected -- and
 * reused by every filtered search on an index of the same device.  On creation the words are uploaded and the
 * ascending list of 128-row tiles that hold a selected row is built on the device (4 bytes per tile), so a filtered
 * search streams only those tiles.  n_rows may be 0 (selects nothing); n_rows < 0, a NULL out, or NULL words with
 * n_rows > 0 are IVR_EINVAL, n_rows above 2^32 IVR_EUNSUPPORTED, all before any device call.  ivr_selection_count
 * returns the number of selected rows (-1 for NULL); ivr_selection_destroy(NULL) is a no-op. */
typedef struct ivr_selection ivr_selection;
IVR_API int     ivr_selection_create(int device, const uint32_t* words_host, int64_t n_rows, ivr_selection** out);
IVR_API int     ivr_selection_destroy(ivr_selection* sel);
IVR_API int64_t ivr_selection_count(const ivr_selection* sel);

/* ivr_index_search / ivr_index_range_search restricted to the selected rows, with the same outputs and semantics:
 * top-k returns the k best selected rows (padded with -1 / -FLT_MAX when fewer are selected), range search every
 * selected row scoring strictly above the radius; ties go to the lower id, a row holding a NaN is never a hit.
 * Selected ids at or past ntotal are ignored.  Both run on the small-batch tcgen05 kernel's filtered variants
 * (search_mma_small_sel_kernel / search_mma_small_sel_range_kernel) for every nq: queries go in chunks of at most 128
 * (fewer where k or the dimension leave less room), and each chunk streams the selected row tiles once.  A selection
 * with no row below ntotal writes the padding (or lims = 0) and launches no scoring kernel.  Errors, before any device
 * call: the argument checks of the unfiltered call, a NULL selection, a search window set on the handle
 * (ivr_index_set_window) and a selection of another device are IVR_EINVAL; an index of 2^32 rows or more, and a dim
 * / k whose 16-query tile does not fit the kernel, are IVR_EUNSUPPORTED.  ivr_index_last_timing reports the filtered
 * call; with several query chunks score_ms runs from the first chunk's scoring to the last one's, prep_ms is the first
 * chunk's and merge_ms the last chunk's. */
IVR_API int ivr_index_search_selected(ivr_index* idx, const ivr_selection* sel, const float* q_host, int64_t nq, int k,
                                      float* D_host, int64_t* I_host);
IVR_API int ivr_index_search_selected_device(ivr_index* idx, const ivr_selection* sel, const float* q_dev, int64_t nq,
                                             int k, float* D_dev, int64_t* I_dev, int64_t id_offset, void* stream);
IVR_API int ivr_index_range_search_selected(ivr_index* idx, const ivr_selection* sel, const float* q_host, int64_t nq,
                                            float radius, int64_t capacity, int64_t* lims_host, float* D_host,
                                            int64_t* I_host);
IVR_API int ivr_index_range_search_selected_device(ivr_index* idx, const ivr_selection* sel, const float* q_dev,
                                                   int64_t nq, float radius, int64_t capacity, int64_t* lims_dev,
                                                   float* D_dev, int64_t* I_dev, int64_t id_offset, void* stream);
/* The filtered searches with the hits left as PACKED exchange keys, the per-rank step of a filtered
 * ShardedFlatIP.search / range_search.  Keys, padding (key 0) and the lims / capacity convention are those of
 * ivr_index_search_keys_device and ivr_index_range_search_keys_device; the semantics are those of the filtered calls
 * above, with ONE difference: these two take the handle's search window (ivr_index_set_window).  The selection is
 * over stored rows; of them only the selected rows inside the window are scored and reported, with ids "stored row +
 * id_offset" (the rows are not renumbered from the window's first row).  A shard that stores its neighbours'
 * boundary rows therefore builds one selection of its stored rows, once, and searches it under whatever window its
 * elastic boundaries give: the window's tiles are cut out of the selection's tile list on the host, without a device
 * sync, and every row of two overlapping shards is reported by the one whose window holds it.  A selection with no
 * selected row inside the window writes key 0 everywhere (or lims = 0) and launches no scoring kernel.  Errors,
 * before any device call: the checks of ivr_index_search_keys_device / ivr_index_range_search_keys_device (including
 * id_offset + ntotal > 2^32: IVR_EUNSUPPORTED) and of the filtered calls above, except that a window is allowed; a
 * window reaching beyond ntotal is IVR_EINVAL.  ivr_index_last_timing reports them as the filtered calls above. */
IVR_API int ivr_index_search_selected_keys_device(ivr_index* idx, const ivr_selection* sel, const float* q_dev,
                                                  int64_t nq, int k, uint64_t* keys_dev, int64_t id_offset,
                                                  void* stream);
IVR_API int ivr_index_range_search_selected_keys_device(ivr_index* idx, const ivr_selection* sel, const float* q_dev,
                                                        int64_t nq, float radius, int64_t capacity,
                                                        int64_t* lims_dev, uint64_t* keys_dev, int64_t id_offset,
                                                        void* stream);

/* Search window: until cleared (count < 0) every search on this handle scores only the stored rows
 * [first, first + count) -- ids are still "stored row + id_offset", k > count pads as usual, a window reaching beyond
 * ntotal fails the search with IVR_EINVAL.  No data moves: this is how a row shard that also holds a replica of its
 * neighbours' boundary rows takes over or gives up rows between two searches (elastic shard boundaries,
 * ShardedFlatIP; no counterpart in the reference, whose shards are whole remote servers: system.py:1715-1757). */
IVR_API int ivr_index_set_window(ivr_index* idx, int64_t first, int64_t count);

/* Kernel timing of the LAST ivr_index_search_device call (CUDA events recorded on
 * the launching stream, only when enabled).  ms[0] = dominant scoring+select kernel,
 * ms[1] = top-k merge kernel(s), ms[2] = query preparation; launches[0..2] = launch
 * counts of the same.  Blocks until those events have completed. */
IVR_API int ivr_index_set_timing(ivr_index* idx, int enable);
IVR_API int ivr_index_last_timing(ivr_index* idx, float ms[3], int launches[3]);
/* which path the last search took (IVR_PATH_STREAM / IVR_PATH_MMA) */
IVR_API int ivr_index_last_path(const ivr_index* idx);
/* name of the dominant scoring kernel of the last search (static string, e.g. "search_mma_xres_kernel") */
IVR_API const char* ivr_index_last_kernel(const ivr_index* idx);

/* K5: merge per-shard top-k lists after the all-gather
 * (semantic precedent: system.py:1721-1746 concat + sort + truncate).
 *   D_parts float32 [n_parts, nq, k], I_parts int64 [n_parts, nq, k] (device),
 *   entries with id < 0 are padding; ids must be below 2^32 (the merge key holds a 32-bit id --
 *   ShardedFlatIP refuses larger indexes).  Output descending, ties -> lower id. */
IVR_API int ivr_topk_merge_device(int device, const float* D_parts, const int64_t* I_parts, int n_parts,
                          int64_t nq, int k, float* D_out, int64_t* I_out, void* stream);
/* The same merge on the packed keys of ivr_index_search_keys_device: keys_parts uint64 [n_parts, nq, k]
 * (device; the all-gather output), n_parts <= 64.  No scratch, no allocation, one kernel launch. */
IVR_API int ivr_topk_merge_keys_device(int device, const uint64_t* keys_parts, int n_parts, int64_t nq, int k,
                               float* D_out, int64_t* I_out, void* stream);
/* Merge of per-part range results (the runs of ivr_index_range_search_keys_device after one all-gather), device:
 *   keys_parts uint64 [n_parts, part_stride]: part p holds query q's hits, sorted (unsigned key descending), at
 *              [lims_parts[p][q], lims_parts[p][q+1])
 *   lims_parts int64  [n_parts, nq + 1]
 * Out: lims int64 [nq + 1], lims[q] = sum over p of lims_parts[p][q]; D float32 / I int64 [lims[nq]] in key order
 * (score descending, then lower id; I = the key's 32-bit id).  An equal key in two parts is placed after the one of
 * the lower part, so the output stays a permutation of the input.  n_parts in 1..64, nq >= 0; keys_parts, D and I
 * may be NULL only when part_stride == 0; else IVR_EINVAL before any device call.  The caller promises
 * part_stride >= lims_parts[p][nq] for every p and monotone lims_parts (they live on the device and are not read
 * back).  Two kernel launches, no atomics, no scratch, no allocation, deterministic. */
IVR_API int ivr_range_merge_keys_device(int device, const uint64_t* keys_parts, int64_t part_stride,
                                        const int64_t* lims_parts, int n_parts, int64_t nq, int64_t* lims, float* D,
                                        int64_t* I, void* stream);

/* ---- K7: cross-shard hit exchange over NVLink / NVSwitch peer memory ------------------------
 * Replaces the "collect every shard's hit list" step of _search_with_remote_index (system.py:1721-1746) for
 * one process per GPU on one box.  Every rank owns a MAILBOX in its HBM: `slots` regions of [world][capacity]
 * packed keys (the format of ivr_index_search_keys_device) + one arrival flag per (slot, sender).
 *   create        allocates and zeroes the mailbox (cudaMalloc, exportable through CUDA IPC)
 *   ipc_handle    64-byte CUDA IPC handle of my mailbox; the caller exchanges the handles of all ranks
 *                 (any control-plane channel, e.g. one torch.distributed all-gather at set-up time)
 *   connect_ipc   maps every peer's mailbox (handles: [world][64] in rank order; my own entry is ignored);
 *                 IVR_EUNSUPPORTED when a peer cannot be mapped (no P2P / different IPC namespace)
 *   connect_ptrs  the same with already-mapped device pointers (ranks living in one process)
 *   push          one kernel: copies my n_entries keys into part `rank` of slot `slot` of EVERY mailbox (16-byte
 *                 peer stores), fences system-wide, then stores `epoch` into my flag of that slot on every rank
 *   wait          queues stream memory operations (cuStreamWaitValue32 >=) until all `world` flags of the slot
 *                 reached `epoch`; no SM is held while waiting
 *   slot          device pointer of the slot: uint64 [world][n_entries] after a completed wait -- the
 *                 keys_parts argument of ivr_topk_merge_keys_device
 * Protocol: search s uses slot s % slots with epoch s / slots + 1; every rank issues push, wait and the merge of
 * consecutive searches in ONE stream, which makes slot reuse safe without acknowledgements (csrc/exchange.cu). */
#define IVR_IPC_HANDLE_BYTES 64
typedef struct ivr_exchange ivr_exchange;
IVR_API int   ivr_exchange_create(int device, int rank, int world, int slots, int64_t capacity, ivr_exchange** out);
IVR_API int   ivr_exchange_destroy(ivr_exchange* ex);
IVR_API void* ivr_exchange_base(ivr_exchange* ex);
IVR_API int   ivr_exchange_ipc_handle(ivr_exchange* ex, uint8_t* handle);
IVR_API int   ivr_exchange_connect_ipc(ivr_exchange* ex, const uint8_t* handles);
IVR_API int   ivr_exchange_connect_ptrs(ivr_exchange* ex, void* const* bases);
IVR_API int   ivr_exchange_push(ivr_exchange* ex, const uint64_t* keys_dev, int64_t n_entries, int slot,
                                uint32_t epoch, void* stream);
IVR_API int   ivr_exchange_wait(ivr_exchange* ex, int slot, uint32_t epoch, void* stream);
IVR_API const uint64_t* ivr_exchange_slot(ivr_exchange* ex, int slot);

/* Replaces faiss.normalize_L2(x) (unified_index.py:1776): in-place row L2
 * normalisation, zero rows untouched. */
IVR_API int ivr_normalize_l2(int device, float* x_host, int64_t n, int d);
IVR_API int ivr_normalize_l2_device(int device, float* x_dev, int64_t n, int d, void* stream);

/* ---- near-duplicate keyframe pruning ------------------------------------
 * All cosines follow sklearn's order of operations (normalise rows, then dot)
 * in fp32, as the reference does through sklearn.metrics.pairwise.
 */

/* Replaces filter.calculate_similarities (filter.py:142-151) and the loop in
 * TemporalAnalyzer.detect_scene_boundaries (core.py:3612-3616):
 *   out[i-1] = cos(e[i-1], e[i]),  i = 1..n-1.   e: float32 [n, d]. */
IVR_API int ivr_consecutive_cosine(int device, const float* e_host, int64_t n, int d, float* out_host);
IVR_API int ivr_consecutive_cosine_device(int device, const float* e_dev, int64_t n, int d,
                                  float* out_dev, void* stream);

/* Replaces filter.filter_similar_frames_advanced applied per scene by
 * filter.apply_similarity_filtering_to_scenes (filter.py:224-259, 261-315):
 * within each inclusive scene [scene_start[s], scene_end[s]] keep the first
 * frame; drop frame i iff some ALREADY KEPT j in [i-min(window,len), i) has
 * cos(e_i, e_j) >= thr.  keep[i] = 1/0; frames outside every scene get 0.
 * Also writes cos_prev[i] = cos(e_i, e_{i-1}) (cos_prev[0] = 1) if non-NULL. */
IVR_API int ivr_dedup_window(int device, const float* e_host, int64_t n, int d,
                     const int64_t* scene_start, const int64_t* scene_end, int64_t n_scenes,
                     int window, float thr, uint8_t* keep_host, float* cos_prev_host);
IVR_API int ivr_dedup_window_device(int device, const float* e_dev, int64_t n, int d,
                            const int64_t* scene_start_dev, const int64_t* scene_end_dev,
                            int64_t n_scenes, int window, float thr,
                            uint8_t* keep_dev, float* cos_prev_dev, uint32_t* mask_ws_dev,
                            void* stream);
/* The whole similarity stage of filter.py in ONE call on host frames -- calculate_similarities ->
 * detect_scene_transitions -> group_into_scenes -> apply_similarity_filtering_to_scenes with
 * filter_similar_frames_advanced (filter.py:142-176, 224-315); what README's FrameFilter.apply_filters names:
 *   e_host   float32 [n, d] raw (un-normalised) frame embeddings.  Page-locked memory is copied from directly;
 *            pageable memory is staged through pinned double buffers by a few host threads.  Either way the
 *            frames cross PCIe ONCE, in 64 MB chunks, each chunk's banded-cosine kernel queued behind its copy.
 *   scenes   frame i starts a scene iff i == 0 or cos(e_i, e_{i-1}) < transition_thr (strict); scenes shorter
 *            than min_scene_len are dropped (keep = 0), exactly like group_into_scenes.
 *   rule     inside a scene keep the first frame; drop frame i iff an already KEPT j in [i - window, i) has
 *            cos(e_i, e_j) >= thr; window <= 0 keeps every frame of every scene (filter.py:233, 242).
 *   outputs  keep_host uint8 [n]; cos_prev_host float32 [n] (cos with the previous frame, [0] = 1) if non-NULL;
 *            stats[0] = scenes that survived the length filter, stats[1] = frames inside them, if non-NULL. */
IVR_API int ivr_frame_filter(int device, const float* e_host, int64_t n, int d, int window, float thr,
                     float transition_thr, int min_scene_len, uint8_t* keep_host, float* cos_prev_host,
                     int64_t stats[2]);

/* Timing of the last ivr_dedup_window_device call on this thread (events on the
 * launching stream): ms[0] = banded-cosine kernel, ms[1] = greedy resolve kernel. */
IVR_API int ivr_dedup_set_timing(int enable);
IVR_API int ivr_dedup_last_timing(float ms[2]);

/* Replaces filter.filter_similar_frames_in_scene (filter.py:178-222) when
 * force_last != 0, and the video_frame_filter.extract_unique_frames rule
 * (video_frame_filter.py:63-70) when force_last == 0 and min_distance == 1:
 * per scene keep frame 0; then keep i iff i - last_kept >= min_distance and
 * cos(e_i, e_last_kept) < thr; with force_last the scene's last frame is kept. */
IVR_API int ivr_dedup_chain(int device, const float* e_host, int64_t n, int d,
                    const int64_t* scene_start, const int64_t* scene_end, int64_t n_scenes,
                    int min_distance, float thr, int force_last, uint8_t* keep_host);

/* Replaces Phase 4 of filter_research_update.AdvancedKeyframeExtractor
 * (filter_research_update.py:316-338): per sequence keep frame 0; keep frame i iff
 * cos(e_i, e_p) < thr for every p in a FIFO of the last `fifo` (1..16, reference: 10) KEPT frames. */
IVR_API int ivr_dedup_fifo(int device, const float* e_host, int64_t n, int d,
                   const int64_t* scene_start, const int64_t* scene_end, int64_t n_scenes,
                   int fifo, float thr, uint8_t* keep_host);

/* ------------------------------------------------------------------------
 * Similar-sequence search (SURVEY.md section 8f, rank 2)
 * ---------------------------------------------------------------------- */
#define IVR_MAX_SEQ_LEN 128

/* Replaces TemporalAnalyzer.find_similar_sequences (core.py:3644-3702, with
 * _compute_sequence_similarity, core.py:3812-3832): for every target window start t in
 * [0, nt - seq_len] and database window start j in [0, nd - seq_len], sim = float32 mean over i of
 * cos(target[t+i], db[j+i]); windows with sim >= threshold are hits.  Host pointers; `target` is
 * float32 [nt, dim], `db` float32 [nd, dim] (raw, un-normalised rows, as the reference passes them).
 * Hits are written UNSORTED to hit_t / hit_j / hit_sim (capacity max_hits each; the host wrapper applies
 * the reference's stable descending sort); *n_hits receives the total number of qualifying windows --
 * when it exceeds max_hits only max_hits of them were stored and the caller retries with larger buffers.
 * nt < seq_len or nd < seq_len yields zero hits (the reference returns [] there). */
IVR_API int ivr_sequence_similarity(int device, const float* target_host, int64_t nt, const float* db_host,
                            int64_t nd, int dim, int seq_len, float threshold, int64_t max_hits,
                            int32_t* hit_t, int64_t* hit_j, float* hit_sim, int64_t* n_hits);

/* eps-neighbourhoods for AdvancedKeyframeExtractor.cluster_similar_frames (filter_research_update.py:113-127:
 * similarity_matrix = cosine_similarity(embeddings); distance = 1 - similarity; DBSCAN(eps, metric='precomputed')).
 * e_host: float32 [n, dim] raw rows; adj_host: uint32 [n, (n + 31) / 32]; bit b of word w of row i is set iff
 * 1 - cos(e_i, e_{32 w + b}) <= eps in float32 (every frame neighbours itself).  The DBSCAN labelling on these
 * bit rows is sequential and done by the host wrapper.  n <= IVR_MAX_CLUSTER_FRAMES. */
#define IVR_MAX_CLUSTER_FRAMES 8192
IVR_API int ivr_cosine_neighbors(int device, const float* e_host, int64_t n, int dim, float eps, uint32_t* adj_host);

/* ------------------------------------------------------------------------
 * .rvdb container: host-side block decoders (SURVEY.md section 8f, rank 1)
 * The reference keeps its embeddings in an HDF5 dataset filtered with shuffle + LZF and its metadata / index
 * blobs as LZ4 frames (unified_index.py:943-956, 1175-1234, 1827-1860).  rvdb_reader.py parses the container;
 * these decode one chunk / block each (plain C on the host, no device involved).
 * ---------------------------------------------------------------------- */
/* liblzf stream -> bytes; returns the decoded size or -1 (malformed input / dst too small) */
IVR_API int64_t ivr_lzf_decompress(const uint8_t* src, int64_t src_len, uint8_t* dst, int64_t dst_cap);
/* one LZ4 block, written at dst + dst_pos (matches may reach back into dst[0, dst_pos): linked blocks of a
 * frame); returns the bytes produced or -1 */
IVR_API int64_t ivr_lz4_block_decompress(const uint8_t* src, int64_t src_len, uint8_t* dst, int64_t dst_pos,
                                 int64_t dst_cap);
/* inverse of the HDF5 shuffle filter (filter id 2) for elements of elem_size bytes */
IVR_API int     ivr_unshuffle(const uint8_t* src, int64_t n_bytes, int elem_size, uint8_t* dst);

#ifdef __cplusplus
}
#endif
#endif /* IVR_B200_H */

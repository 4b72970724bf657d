// capi.cu -- the extern "C" surface declared in include/ivr_b200.h.
#include "index.cuh"

#include <algorithm>
#include <climits>
#include <cstdarg>
#include <cstring>
#include <new>
#include <thread>
#include <vector>

namespace ivr {

// Pageable host memory <-> pinned staging.  One thread moves ~5-8 GB/s, a PCIe 5 x16 link ~50 GB/s: large blocks
// are split over a few threads so that the staging copy does not throttle the H2D stream behind it.
static void staged_memcpy(void* dst, const void* src, size_t bytes) {
    constexpr size_t kMinPerThread = static_cast<size_t>(4) << 20;
    unsigned hw = std::thread::hardware_concurrency();
    size_t nt = std::min<size_t>({static_cast<size_t>(8), hw ? hw : 1, bytes / kMinPerThread});
    if (nt <= 1) { memcpy(dst, src, bytes); return; }
    std::vector<std::thread> th;
    const size_t per = (bytes / nt + 4095) & ~static_cast<size_t>(4095);
    for (size_t t = 1; t < nt; ++t) {
        const size_t o = t * per;
        if (o >= bytes) break;
        const size_t len = std::min(per, bytes - o);
        th.emplace_back([=] { memcpy(static_cast<char*>(dst) + o, static_cast<const char*>(src) + o, len); });
    }
    memcpy(dst, src, std::min(per, bytes));
    for (auto& t : th) t.join();
}

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// other translation units
int convert_rows(ivr_index* idx, const float* src_dev, int64_t n, int64_t dst_row, cudaStream_t st);
int normalize_l2_device(float* x_dev, int64_t n, int d, cudaStream_t st);
int reconstruct_rows(ivr_index* idx, int64_t first, int64_t n, float* dst_dev, cudaStream_t st);
int pack_parts(const float* D, const int64_t* I, uint64_t* keys, int64_t n, cudaStream_t st);
int dedup_set_timing(int enable);
int dedup_last_timing(float ms[2]);
int launch_banded(const float* e_dev, int64_t n, int64_t out_begin, int d, int window, float thr, uint32_t* masks,
                  float* cos_prev, int sm_count, cudaStream_t st);
int launch_scene_resolve(const uint32_t* masks, const float* cos_prev, int64_t n, int window, float transition_thr,
                         int min_len, uint8_t* keep, unsigned long long* stats, cudaStream_t st);
int dedup_window_device(int device, const float* e_dev, int64_t n, int d,
                        const int64_t* scene_start_dev, const int64_t* scene_end_dev,
                        int64_t n_scenes, int window, float thr, uint8_t* keep_dev,
                        float* cos_prev_dev, uint32_t* mask_ws_dev, cudaStream_t st);
int dedup_chain_device(const float* e_dev, int64_t n, int d, const int64_t* scene_start_dev,
                       const int64_t* scene_end_dev, int64_t n_scenes, int min_distance, float thr,
                       int force_last, int fifo, uint8_t* keep_dev, cudaStream_t st);

int sequence_similarity_device(const float* target, int64_t nt, const float* db, int64_t nd, int dim, int seq_len,
                               float thr, int64_t max_hits, int32_t* hit_t, int64_t* hit_j, float* hit_sim,
                               unsigned long long* n_hits_dev, float* tn, float* dn, float* cblock,
                               int64_t block_cols, cudaStream_t st);
int64_t sequence_block_cols(int64_t nt, int64_t nd, int seq_len);
int cosine_neighbors_device(const float* e, int n, int dim, float eps, float* xn, float* cmat, uint32_t* adj,
                            cudaStream_t st);

static int require_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        set_error("no CUDA device available (%s); this library has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return IVR_ENODEVICE;
    }
    if (device < 0 || device >= n) {
        set_error("device %d out of range (have %d)", device, n);
        return IVR_EINVAL;
    }
    int major = 0;
    IVR_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) {
        set_error("device %d has compute capability %d.x; kernels are built for sm_100a only", device, major);
        return IVR_ENODEVICE;
    }
    IVR_CUDA(cudaSetDevice(device));
    static bool pool_kept[64] = {};
    if (device < 64 && !pool_kept[device]) {                        // keep freed blocks in the pool (see DevBuf)
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t never = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &never);
        }
        cudaGetLastError();
        pool_kept[device] = true;
    }
    return IVR_OK;
}

// require_device() with its capability probe done once per thread and device, for entry points called per search
static int require_device_once(int device) {
    static thread_local int checked_device = -1;
    if (checked_device == device) { IVR_CUDA(cudaSetDevice(device)); return IVR_OK; }
    IVR_TRY(require_device(device));
    checked_device = device;
    return IVR_OK;
}

// Scoped device buffer for the host-pointer dedup / normalise entry points.  Stream-ordered allocation from the
// device's default memory pool, whose release threshold require_device() raises to "never": after the first call
// the blocks come back from the pool without a driver allocation (a cudaMalloc / cudaFree pair per call used to cost
// more than the kernels they served).
struct DevBuf {
    void* p = nullptr;
    cudaStream_t st = nullptr;
    ~DevBuf() { if (p) cudaFreeAsync(p, st); }
    int alloc(size_t bytes, cudaStream_t stream = nullptr) {
        st = stream;
        IVR_CUDA(cudaMallocAsync(&p, bytes ? bytes : 1, st));
        return IVR_OK;
    }
};

}  // namespace ivr

using namespace ivr;

extern "C" {

const char* ivr_last_error(void) { return g_err; }
int ivr_version(void) { return 100; }

int ivr_device_count(int* count) {
    if (!count) { set_error("count is NULL"); return IVR_EINVAL; }
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { cudaGetLastError(); n = 0; }
    *count = n;
    return IVR_OK;
}

int ivr_device_info(int device, char* name, size_t name_len, int* sm_count, int* cc_major,
                    int* cc_minor, size_t* total_bytes) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) {
        cudaGetLastError();
        set_error("device %d not available", device);
        return IVR_ENODEVICE;
    }
    cudaDeviceProp p;
    IVR_CUDA(cudaGetDeviceProperties(&p, device));
    if (name && name_len) { strncpy(name, p.name, name_len - 1); name[name_len - 1] = 0; }
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (total_bytes) *total_bytes = p.totalGlobalMem;
    return IVR_OK;
}

// ---------------------------------------------------------------- index ----
int ivr_index_create(int dim, int device, ivr_index** out) {
    if (!out) { set_error("out is NULL"); return IVR_EINVAL; }
    *out = nullptr;
    if (dim <= 0 || dim > 8192) { set_error("dim %d out of range (1..8192)", dim); return IVR_EINVAL; }
    IVR_TRY(require_device(device));
    ivr_index* idx = new (std::nothrow) ivr_index();
    if (!idx) { set_error("out of host memory"); return IVR_ENOMEM; }
    idx->dim = dim;
    idx->dpad = pad_dim(dim);
    idx->device = device;
    cudaError_t e = cudaDeviceGetAttribute(&idx->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&idx->stream, cudaStreamNonBlocking);
    for (int i = 0; i < 6 && e == cudaSuccess; ++i) e = cudaEventCreate(&idx->ev[i]);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&idx->rows_ready, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&idx->sel_state), 256);
    if (e == cudaSuccess) e = cudaMemset(idx->sel_state, 0, 256);
    if (e != cudaSuccess) {
        set_error("index_create: %s", cudaGetErrorString(e));
        delete idx;
        return IVR_ECUDA;
    }
    *out = idx;
    return IVR_OK;
}

int ivr_index_destroy(ivr_index* idx) {
    if (!idx) return IVR_OK;
    cudaSetDevice(idx->device);
    cudaDeviceSynchronize();
    if (idx->rows) cudaFree(idx->rows);
    if (idx->ws) cudaFree(idx->ws);
    if (idx->io) cudaFree(idx->io);
    if (idx->sel_state) cudaFree(idx->sel_state);
    if (idx->pin) cudaFreeHost(idx->pin);
    for (auto& ev : idx->ev) if (ev) cudaEventDestroy(ev);
    if (idx->rows_ready) cudaEventDestroy(idx->rows_ready);
    if (idx->stream) cudaStreamDestroy(idx->stream);
    delete idx;
    return IVR_OK;
}

int ivr_index_reserve(ivr_index* idx, int64_t n_rows) {
    if (!idx || n_rows < 0) { set_error("reserve: bad argument"); return IVR_EINVAL; }
    if (n_rows > 0x7fffffff) { set_error("a shard holds at most 2^31-1 rows"); return IVR_EUNSUPPORTED; }
    IVR_CUDA(cudaSetDevice(idx->device));
    return ensure_capacity(idx, n_rows, idx->stream, /*exact=*/true);
}

int ivr_index_add_device(ivr_index* idx, const float* x_dev, int64_t n, void* stream) {
    if (!idx || n < 0 || (n > 0 && !x_dev)) { set_error("add_device: bad argument"); return IVR_EINVAL; }
    if (n == 0) return IVR_OK;
    IVR_CUDA(cudaSetDevice(idx->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);       // NULL = the legacy default stream, as in CUDA
    if (idx->ntotal + n > 0x7fffffff) { set_error("a shard holds at most 2^31-1 rows"); return IVR_EUNSUPPORTED; }
    IVR_TRY(ensure_capacity(idx, idx->ntotal + n, st));
    IVR_TRY(convert_rows(idx, x_dev, n, idx->ntotal, st));
    IVR_CUDA(cudaEventRecord(idx->rows_ready, st));
    idx->rows_ready_set = true;
    idx->ntotal += n;
    return IVR_OK;
}

int ivr_index_add(ivr_index* idx, const float* x_host, int64_t n) {
    if (!idx || n < 0 || (n > 0 && !x_host)) { set_error("add: bad argument"); return IVR_EINVAL; }
    if (n == 0) return IVR_OK;
    IVR_CUDA(cudaSetDevice(idx->device));
    if (idx->ntotal + n > 0x7fffffff) { set_error("a shard holds at most 2^31-1 rows"); return IVR_EUNSUPPORTED; }
    cudaStream_t st = idx->stream;
    IVR_TRY(ensure_capacity(idx, idx->ntotal + n, st));
    // stage through two pinned half-buffers + a device fp32 staging area in the workspace
    const size_t row_bytes = static_cast<size_t>(idx->dim) * sizeof(float);
    int64_t chunk = std::max<int64_t>(1, (static_cast<int64_t>(32) << 20) / static_cast<int64_t>(row_bytes));
    chunk = std::min(chunk, n);
    IVR_TRY(ensure_pin(idx, 2 * chunk * row_bytes));
    IVR_TRY(ensure_ws(idx, 2 * chunk * row_bytes));
    cudaEvent_t done[2] = {nullptr, nullptr};
    for (auto& e : done)
        if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) {
            if (done[0]) cudaEventDestroy(done[0]);
            set_error("add: cudaEventCreate failed");
            return IVR_ECUDA;
        }
    int rc = IVR_OK;
    int64_t off = 0;
    for (int it = 0; off < n; ++it) {
        const int64_t m = std::min(chunk, n - off);
        const int b = it & 1;
        char* pin = static_cast<char*>(idx->pin) + b * chunk * row_bytes;
        float* dev = reinterpret_cast<float*>(static_cast<char*>(idx->ws) + b * chunk * row_bytes);
        if (it >= 2 && cudaEventSynchronize(done[b]) != cudaSuccess) { rc = IVR_ECUDA; break; }
        staged_memcpy(pin, x_host + off * idx->dim, m * row_bytes);
        if (cudaMemcpyAsync(dev, pin, m * row_bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) { rc = IVR_ECUDA; break; }
        rc = convert_rows(idx, dev, m, idx->ntotal + off, st);
        if (rc != IVR_OK) break;
        cudaEventRecord(done[b], st);
        off += m;
    }
    cudaError_t e = cudaStreamSynchronize(st);
    for (auto& ev : done) cudaEventDestroy(ev);
    if (rc == IVR_OK && e != cudaSuccess) { set_error("add: %s", cudaGetErrorString(e)); rc = IVR_ECUDA; }
    if (rc == IVR_ECUDA && g_err[0] == 0) set_error("add: CUDA failure");
    if (rc == IVR_OK) idx->ntotal += n;                          // the stream was drained above: rows are visible to every stream
    return rc;
}

int ivr_index_reconstruct(ivr_index* idx, int64_t first, int64_t n, float* x_host) {
    if (!idx || first < 0 || n < 0 || (n > 0 && !x_host)) { set_error("reconstruct: bad argument"); return IVR_EINVAL; }
    if (first + n > idx->ntotal) {
        set_error("reconstruct: rows [%lld, %lld) outside the %lld stored", static_cast<long long>(first),
                  static_cast<long long>(first + n), static_cast<long long>(idx->ntotal));
        return IVR_EINVAL;
    }
    if (n == 0) return IVR_OK;
    IVR_CUDA(cudaSetDevice(idx->device));
    cudaStream_t st = idx->stream;
    if (idx->rows_ready_set) IVR_CUDA(cudaStreamWaitEvent(st, idx->rows_ready, 0));
    // fp16 -> fp32 on the device, then D2H through the two pinned half-buffers (the mirror image of ivr_index_add)
    const size_t row_bytes = static_cast<size_t>(idx->dim) * sizeof(float);
    int64_t chunk = std::max<int64_t>(1, (static_cast<int64_t>(32) << 20) / static_cast<int64_t>(row_bytes));
    chunk = std::min(chunk, n);
    IVR_TRY(ensure_pin(idx, 2 * chunk * row_bytes));
    IVR_TRY(ensure_ws(idx, 2 * chunk * row_bytes));
    cudaEvent_t done[2] = {nullptr, nullptr};
    for (auto& e : done)
        if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) {
            if (done[0]) cudaEventDestroy(done[0]);
            set_error("reconstruct: cudaEventCreate failed");
            return IVR_ECUDA;
        }
    int rc = IVR_OK;
    int64_t off = 0, prev_off = 0, prev_m = 0;
    for (int it = 0; ; ++it) {
        const int b = it & 1;
        int64_t m = 0;
        if (off < n) {                                                 // queue chunk `it` ...
            m = std::min(chunk, n - off);
            char* pin = static_cast<char*>(idx->pin) + b * chunk * row_bytes;
            float* dev = reinterpret_cast<float*>(static_cast<char*>(idx->ws) + b * chunk * row_bytes);
            rc = reconstruct_rows(idx, first + off, m, dev, st);
            if (rc != IVR_OK) break;
            if (cudaMemcpyAsync(pin, dev, m * row_bytes, cudaMemcpyDeviceToHost, st) != cudaSuccess) { rc = IVR_ECUDA; break; }
            cudaEventRecord(done[b], st);
        }
        if (it > 0) {                                                  // ... while chunk `it - 1` is copied out
            const int pb = (it - 1) & 1;
            if (cudaEventSynchronize(done[pb]) != cudaSuccess) { rc = IVR_ECUDA; break; }
            staged_memcpy(x_host + prev_off * idx->dim, static_cast<char*>(idx->pin) + pb * chunk * row_bytes, prev_m * row_bytes);
        }
        if (off >= n) break;
        prev_off = off; prev_m = m;
        off += m;
    }
    cudaError_t e = cudaStreamSynchronize(st);
    for (auto& ev : done) cudaEventDestroy(ev);
    if (rc == IVR_OK && e != cudaSuccess) { set_error("reconstruct: %s", cudaGetErrorString(e)); rc = IVR_ECUDA; }
    if (rc == IVR_ECUDA && g_err[0] == 0) set_error("reconstruct: CUDA failure");
    return rc;
}

int ivr_index_reset(ivr_index* idx) {
    if (!idx) { set_error("reset: NULL index"); return IVR_EINVAL; }
    idx->ntotal = 0;
    return IVR_OK;
}

int ivr_index_set_window(ivr_index* idx, int64_t first, int64_t count) {
    if (!idx) { set_error("set_window: NULL index"); return IVR_EINVAL; }
    if (count < 0) { idx->win_first = 0; idx->win_count = -1; return IVR_OK; }
    if (first < 0) { set_error("set_window: first row must be >= 0 (got %lld)", static_cast<long long>(first)); return IVR_EINVAL; }
    idx->win_first = first;
    idx->win_count = count;
    return IVR_OK;
}

int64_t ivr_index_ntotal(const ivr_index* idx) { return idx ? idx->ntotal : -1; }
int ivr_selection_create(int device, const uint32_t* words_host, int64_t n_rows, ivr_selection** out) {
    if (!out) { set_error("selection_create: out is NULL"); return IVR_EINVAL; }
    *out = nullptr;
    if (n_rows < 0) {
        set_error("selection_create: n_rows must be >= 0 (got %lld)", static_cast<long long>(n_rows));
        return IVR_EINVAL;
    }
    if (n_rows > 0 && !words_host) { set_error("selection_create: words is NULL"); return IVR_EINVAL; }
    if (n_rows > (1ll << 32)) {
        set_error("selection_create: row ids must stay below 2^32 (got %lld rows)", static_cast<long long>(n_rows));
        return IVR_EUNSUPPORTED;
    }
    IVR_TRY(require_device(device));
    return selection_create(device, words_host, n_rows, out);
}

int ivr_selection_destroy(ivr_selection* sel) { return selection_destroy(sel); }
int64_t ivr_selection_count(const ivr_selection* sel) { return sel ? sel->count : -1; }

int ivr_index_dim(const ivr_index* idx) { return idx ? idx->dim : -1; }
int ivr_index_device(const ivr_index* idx) { return idx ? idx->device : -1; }

// --------------------------------------------------------------- search ----
__global__ void fill_empty_kernel(float* D, int64_t* I, int64_t n) {
    const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (i >= n) return;
    if (D) { D[i] = -3.402823466e+38f; I[i] = -1; }
    else I[i] = 0;                                   // packed-key output: key 0 = padding
}

}  // extern "C"

namespace ivr {

// Which kernel family serves (nq, k) on this index.  IVR_PATH_AUTO: ONE query streams on the SIMT kernel; from two
// queries up the tcgen05 kernels win -- the small-batch kernel wherever its resident query tile fits (any dimension),
// the batched kernels up to 1024 dims.  (Two queries on the streaming kernel are shared-memory bound: 0.27 / 0.79 /
// 2.08 / 17.9 ms at 1 / 3 / 10 / 100 M x 512 rows against 0.26 / 0.60 / 1.75 / 14.8 ms on the small-batch kernel,
// which serves small shards in its one-launch dump mode.)  Shapes neither tcgen05 kernel fits (e.g. dim > 1024 with a
// large batch) stream.
static int choose_path(const ivr_index* idx, int64_t nq, int k, int path) {
    const bool small_ok = mma_small_supported(idx, nq, k), big_ok = mma_supported(idx, nq, k);
    if (path == IVR_PATH_AUTO) {
        // IVR_AUTO_STREAM_MAX_NQ: tuning knob (measurements only) -- largest batch the streaming kernel serves
        const char* e = getenv("IVR_AUTO_STREAM_MAX_NQ");
        const int64_t stream_max = (e && *e) ? atoi(e) : 1;
        if (nq <= stream_max) return IVR_PATH_STREAM;
        return (small_ok || big_ok) ? IVR_PATH_MMA : IVR_PATH_STREAM;
    }
    if (path == IVR_PATH_MMA && !small_ok && !big_ok) {
        set_error("search: the tcgen05 path does not support dim=%d nq=%lld k=%d", idx->dim,
                  static_cast<long long>(nq), k);
        return IVR_EUNSUPPORTED;
    }
    if (path != IVR_PATH_MMA && path != IVR_PATH_STREAM) { set_error("search: unknown path %d", path); return IVR_EINVAL; }
    return path;
}

// While alive, the search back-ends see only the rows of the handle's search window (ivr_index_set_window): the row
// block starts at the window's first row and holds win_count rows; reported ids are shifted back by the caller.
struct RowWindow {
    ivr_index* idx;
    __half*    rows;
    int64_t    ntotal, capacity;
    explicit RowWindow(ivr_index* i) : idx(i), rows(i->rows), ntotal(i->ntotal), capacity(i->capacity) {
        if (idx->win_count < 0) return;
        idx->rows = rows + idx->win_first * idx->dpad;
        idx->ntotal = idx->win_count;
        idx->capacity = capacity - idx->win_first;
    }
    ~RowWindow() { idx->rows = rows; idx->ntotal = ntotal; idx->capacity = capacity; }
};

// The preamble of every query over the stored rows: runs body(id_offset) on the rows of the handle's search window
// (ivr_index_set_window; ids stay "stored row + id_offset") after the rows added on other streams.  `who` prefixes
// the error message.
template <class Body>
static int with_search_window(ivr_index* idx, int64_t id_offset, cudaStream_t st, const char* who, Body&& body) {
    if (idx->win_count >= 0) {
        if (idx->win_first + idx->win_count > idx->ntotal) {
            set_error("%s: the window [%lld, +%lld) reaches beyond the %lld rows of the index", who,
                      static_cast<long long>(idx->win_first), static_cast<long long>(idx->win_count),
                      static_cast<long long>(idx->ntotal));
            return IVR_EINVAL;
        }
        id_offset += idx->win_first;
    }
    RowWindow window(idx);
    IVR_CUDA(cudaSetDevice(idx->device));
    if (idx->rows_ready_set) IVR_CUDA(cudaStreamWaitEvent(st, idx->rows_ready, 0));   // rows added on another stream
    return body(id_offset);
}

// D_dev == nullptr selects the packed-key output: I_dev then receives uint64 keys [nq, k]
// (order_preserving(score) << 32 | ~(row + id_offset), 0 = padding) instead of int64 ids.
static int search_device_impl(ivr_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev,
                              int64_t* I_dev, int64_t id_offset, int path, cudaStream_t st) {
    if (k <= 0) { set_error("search: k must be positive (got %d)", k); return IVR_EINVAL; }
    if (k > IVR_MAX_K) { set_error("search: k=%d exceeds IVR_MAX_K=%d", k, IVR_MAX_K); return IVR_EUNSUPPORTED; }
    if (nq == 0) return IVR_OK;
    return with_search_window(idx, id_offset, st, "search", [&](int64_t id_offset) {
        idx->launches[0] = idx->launches[1] = idx->launches[2] = 0;
        idx->ev_valid[0] = idx->ev_valid[1] = idx->ev_valid[2] = false;
        if (idx->ntotal == 0) {
            const int64_t n = nq * k;
            fill_empty_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(D_dev, I_dev, n);
            IVR_CUDA(cudaGetLastError());
            idx->last_path = 0;
            return IVR_OK;
        }
        const int use = choose_path(idx, nq, k, path);
        if (use < 0) return use;
        if (use == IVR_PATH_MMA) {
            idx->last_path = IVR_PATH_MMA;
            return search_mma(idx, q_dev, nq, k, D_dev, I_dev, id_offset, st);
        }
        idx->last_path = IVR_PATH_STREAM;
        idx->last_kernel = "search_stream_kernel";
        return search_stream(idx, q_dev, nq, k, D_dev, I_dev, id_offset, st);
    });
}

// Checks of ivr_index_range_search*(), in an order that needs no device.
static int range_args(const ivr_index* idx, const void* q, int64_t nq, float radius, int64_t capacity,
                      const void* lims, const void* D, const void* I) {
    if (nq < 0) { set_error("range_search: nq must be >= 0 (got %lld)", static_cast<long long>(nq)); return IVR_EINVAL; }
    if (capacity < 0) {
        set_error("range_search: capacity must be >= 0 (got %lld)", static_cast<long long>(capacity));
        return IVR_EINVAL;
    }
    if (radius != radius) { set_error("range_search: radius is NaN"); return IVR_EINVAL; }
    if (!idx || !lims || (nq > 0 && !q) || (capacity > 0 && (!D || !I))) {
        set_error("range_search: bad argument (NULL index or buffer)");
        return IVR_EINVAL;
    }
    if (capacity > INT_MAX || nq >= INT_MAX) {
        set_error("range_search: at most 2^31-1 hits and queries per call (capacity %lld, nq %lld)",
                  static_cast<long long>(capacity), static_cast<long long>(nq));
        return IVR_EUNSUPPORTED;
    }
    if (small_range_chunk(idx) < 16) {
        set_error("range_search: dim %d is wider than the small-batch kernel holds (padded dim <= 4096)", idx->dim);
        return IVR_EUNSUPPORTED;
    }
    if (idx->ntotal >= (1ll << 32)) {
        set_error("range_search: the hit key holds a 32-bit row; the index has %lld rows",
                  static_cast<long long>(idx->ntotal));
        return IVR_EUNSUPPORTED;
    }
    return IVR_OK;
}

// Checks of ivr_index_range_self_join*(), in an order that needs no device.  The join covers the rows of the search
// window; their count is the number of CUB segments, an int.
static int join_args(const ivr_index* idx, float radius, int64_t capacity, const void* lims, const void* D,
                     const void* I) {
    if (radius != radius) { set_error("range_self_join: radius is NaN"); return IVR_EINVAL; }
    if (capacity < 0) {
        set_error("range_self_join: capacity must be >= 0 (got %lld)", static_cast<long long>(capacity));
        return IVR_EINVAL;
    }
    if (!idx || !lims || (capacity > 0 && (!D || !I))) {
        set_error("range_self_join: bad argument (NULL index or buffer)");
        return IVR_EINVAL;
    }
    if (capacity > INT_MAX) {
        set_error("range_self_join: at most 2^31-1 hits per call (capacity %lld)", static_cast<long long>(capacity));
        return IVR_EUNSUPPORTED;
    }
    if (small_range_chunk(idx) < 16) {
        set_error("range_self_join: dim %d is wider than the small-batch kernel holds (padded dim <= 4096)", idx->dim);
        return IVR_EUNSUPPORTED;
    }
    if (idx->ntotal >= (1ll << 32)) {
        set_error("range_self_join: the hit key holds a 32-bit row; the index has %lld rows",
                  static_cast<long long>(idx->ntotal));
        return IVR_EUNSUPPORTED;
    }
    if ((idx->win_count >= 0 ? idx->win_count : idx->ntotal) >= INT_MAX) {
        set_error("range_self_join: at most 2^31-2 rows per join (window of %lld rows)",
                  static_cast<long long>(idx->win_count));
        return IVR_EUNSUPPORTED;
    }
    return IVR_OK;
}

// Checks shared by the filtered entry points (ivr_index_*_selected*), in an order that needs no device; `windowed`:
// the call honours the handle's search window (the *_selected_keys_device calls), else a window is refused.
static int selected_args(const ivr_index* idx, const ivr_selection* sel, const char* who, bool windowed = false) {
    if (!idx || !sel) { set_error("%s: bad argument (NULL index or selection)", who); return IVR_EINVAL; }
    if (!windowed && idx->win_count >= 0) {
        set_error("%s: the index has a search window; filtered search covers all stored rows (clear the window with "
                  "ivr_index_set_window(idx, 0, -1), or select only the window's rows)", who);
        return IVR_EINVAL;
    }
    if (sel->device != idx->device) {
        set_error("%s: the selection lives on device %d, the index on device %d", who, sel->device, idx->device);
        return IVR_EINVAL;
    }
    if (idx->ntotal >= (1ll << 32)) {
        set_error("%s: filtered search reports 32-bit rows; the index has %lld rows", who,
                  static_cast<long long>(idx->ntotal));
        return IVR_EUNSUPPORTED;
    }
    return IVR_OK;
}

// The preamble of the filtered calls that honour the search window (ivr_index_*_selected_keys_device): body(cut) runs
// on the selected rows of the window, or of every stored row, after the rows added on other streams.  The selection is
// over stored rows, so the rows are not shifted (RowWindow): the window's tiles are cut out of the selection's list on
// the host and ids stay "stored row + id_offset".  A window reaching past the rows is IVR_EINVAL before any device call.
template <class Body>
static int with_selected_window(ivr_index* idx, const ivr_selection* sel, cudaStream_t st, const char* who,
                                Body&& body) {
    int64_t first = 0, end = idx->ntotal;
    if (idx->win_count >= 0) {
        if (idx->win_first + idx->win_count > idx->ntotal) {
            set_error("%s: the window [%lld, +%lld) reaches beyond the %lld rows of the index", who,
                      static_cast<long long>(idx->win_first), static_cast<long long>(idx->win_count),
                      static_cast<long long>(idx->ntotal));
            return IVR_EINVAL;
        }
        first = idx->win_first;
        end = first + idx->win_count;
    }
    IVR_CUDA(cudaSetDevice(idx->device));
    if (idx->rows_ready_set) IVR_CUDA(cudaStreamWaitEvent(st, idx->rows_ready, 0));   // rows added on another stream
    return body(selection_cut(sel, first, end));
}

// ivr_index_search_selected_device after the pointer checks: the top-k of the selected rows, on the filtered
// small-batch kernel; no selected row below ntotal (or no row) writes the padding and scores nothing.  `windowed`: the
// selected rows of the search window only (ivr_index_search_selected_keys_device).  D_dev == nullptr: packed keys.
static int search_selected_impl(ivr_index* idx, const ivr_selection* sel, const float* q_dev, int64_t nq, int k,
                                float* D_dev, int64_t* I_dev, int64_t id_offset, cudaStream_t st,
                                const char* who = "search_selected", bool windowed = false) {
    if (k <= 0) { set_error("%s: k must be positive (got %d)", who, k); return IVR_EINVAL; }
    if (k > IVR_MAX_K) { set_error("%s: k=%d exceeds IVR_MAX_K=%d", who, k, IVR_MAX_K); return IVR_EUNSUPPORTED; }
    IVR_TRY(selected_args(idx, sel, who, windowed));
    if (small_sel_chunk(idx, k) == 0) {
        set_error("%s: dim %d with k=%d does not fit one 16-query tile of the small-batch kernel", who, idx->dim, k);
        return IVR_EUNSUPPORTED;
    }
    if (nq == 0) return IVR_OK;
    auto run = [&](const SelCut& cut, int64_t id_offset) {
        idx->launches[0] = idx->launches[1] = idx->launches[2] = 0;
        idx->ev_valid[0] = idx->ev_valid[1] = idx->ev_valid[2] = false;
        if (cut.n_tiles == 0) {
            const int64_t n = nq * k;
            fill_empty_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(D_dev, I_dev, n);
            IVR_CUDA(cudaGetLastError());
            idx->last_path = 0;
            return IVR_OK;
        }
        idx->last_path = IVR_PATH_MMA;
        return search_mma_small_selected(idx, cut, q_dev, nq, k, D_dev, I_dev, id_offset, st);
    };
    if (windowed)
        return with_selected_window(idx, sel, st, who, [&](const SelCut& cut) { return run(cut, id_offset); });
    return with_search_window(idx, id_offset, st, who, [&](int64_t id_offset) {
        return run(selection_all(sel, idx->ntotal), id_offset);
    });
}

// Exchange keys hold a 32-bit row: the global ids id_offset + [0, ntotal) must fit.
static int check_key_ids(const ivr_index* idx, int64_t id_offset, const char* who) {
    if (id_offset < 0 || id_offset + idx->ntotal > 0x100000000ll) {
        set_error("%s: global row ids must stay below 2^32 (offset %lld + %lld rows)", who,
                  static_cast<long long>(id_offset), static_cast<long long>(idx->ntotal));
        return IVR_EUNSUPPORTED;
    }
    return IVR_OK;
}

}  // namespace ivr

extern "C" {

int ivr_index_search_device(ivr_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev,
                            int64_t* I_dev, int64_t id_offset, int path, void* stream) {
    if (!idx || nq < 0 || (nq > 0 && (!q_dev || !D_dev || !I_dev))) {
        set_error("search: bad argument");
        return IVR_EINVAL;
    }
    // NULL = the legacy default stream, as in CUDA
    return search_device_impl(idx, q_dev, nq, k, D_dev, I_dev, id_offset, path, static_cast<cudaStream_t>(stream));
}

int ivr_index_search_keys_device(ivr_index* idx, const float* q_dev, int64_t nq, int k, uint64_t* keys_dev,
                                 int64_t id_offset, int path, void* stream) {
    if (!idx || nq < 0 || (nq > 0 && (!q_dev || !keys_dev))) {
        set_error("search_keys: bad argument");
        return IVR_EINVAL;
    }
    IVR_TRY(check_key_ids(idx, id_offset, "search_keys"));
    return search_device_impl(idx, q_dev, nq, k, nullptr, reinterpret_cast<int64_t*>(keys_dev), id_offset, path,
                              static_cast<cudaStream_t>(stream));
}

}  // extern "C"

namespace ivr {

// The host-pointer top-k searches: queries in and D / I out through the handle's pinned and device staging buffers,
// device_call(q_dev, D_dev, I_dev, stream) in between.
template <class DeviceCall>
static int host_search(ivr_index* idx, const float* q_host, int64_t nq, int k, float* D_host, int64_t* I_host,
                       DeviceCall&& device_call) {
    if (!idx || nq < 0 || (nq > 0 && (!q_host || !D_host || !I_host))) {
        set_error("search: bad argument");
        return IVR_EINVAL;
    }
    if (k <= 0) { set_error("search: k must be positive (got %d)", k); return IVR_EINVAL; }
    if (k > IVR_MAX_K) { set_error("search: k=%d exceeds IVR_MAX_K=%d", k, IVR_MAX_K); return IVR_EUNSUPPORTED; }
    if (nq == 0) return IVR_OK;
    IVR_CUDA(cudaSetDevice(idx->device));
    cudaStream_t st = idx->stream;
    const size_t qb = static_cast<size_t>(nq) * idx->dim * sizeof(float);
    const size_t db = static_cast<size_t>(nq) * k * sizeof(float);
    const size_t ib = static_cast<size_t>(nq) * k * sizeof(int64_t);
    Carve carve;                                                    // the same layout in the pinned and the device buffer
    const size_t o_q = carve(qb), o_d = carve(db), o_i = carve(ib);
    IVR_TRY(ensure_pin(idx, carve.size));
    char* pin = static_cast<char*>(idx->pin);
    IVR_TRY(ensure_io(idx, carve.size));
    char* io = static_cast<char*>(idx->io);
    float* dq = reinterpret_cast<float*>(io + o_q);
    float* dd = reinterpret_cast<float*>(io + o_d);
    int64_t* di = reinterpret_cast<int64_t*>(io + o_i);
    memcpy(pin + o_q, q_host, qb);
    IVR_CUDA(cudaMemcpyAsync(dq, pin + o_q, qb, cudaMemcpyHostToDevice, st));
    IVR_TRY(device_call(dq, dd, di, st));
    IVR_CUDA(cudaMemcpyAsync(pin + o_d, dd, db, cudaMemcpyDeviceToHost, st));
    IVR_CUDA(cudaMemcpyAsync(pin + o_i, di, ib, cudaMemcpyDeviceToHost, st));
    IVR_CUDA(cudaStreamSynchronize(st));
    memcpy(D_host, pin + o_d, db);
    memcpy(I_host, pin + o_i, ib);
    return IVR_OK;
}

}  // namespace ivr

extern "C" {

int ivr_index_search(ivr_index* idx, const float* q_host, int64_t nq, int k, float* D_host,
                     int64_t* I_host, int path) {
    return host_search(idx, q_host, nq, k, D_host, I_host, [&](const float* dq, float* dd, int64_t* di, cudaStream_t st) {
        return search_device_impl(idx, dq, nq, k, dd, di, 0, path, st);
    });
}

int ivr_index_search_selected_device(ivr_index* idx, const ivr_selection* sel, const float* q_dev, int64_t nq, int k,
                                     float* D_dev, int64_t* I_dev, int64_t id_offset, void* stream) {
    if (!idx || nq < 0 || (nq > 0 && (!q_dev || !D_dev || !I_dev))) {
        set_error("search_selected: bad argument");
        return IVR_EINVAL;
    }
    return search_selected_impl(idx, sel, q_dev, nq, k, D_dev, I_dev, id_offset, static_cast<cudaStream_t>(stream));
}

int ivr_index_search_selected(ivr_index* idx, const ivr_selection* sel, const float* q_host, int64_t nq, int k,
                              float* D_host, int64_t* I_host) {
    IVR_TRY(selected_args(idx, sel, "search_selected"));
    return host_search(idx, q_host, nq, k, D_host, I_host, [&](const float* dq, float* dd, int64_t* di, cudaStream_t st) {
        return search_selected_impl(idx, sel, dq, nq, k, dd, di, 0, st);
    });
}

int ivr_index_range_search_device(ivr_index* idx, const float* q_dev, int64_t nq, float radius, int64_t capacity,
                                  int64_t* lims_dev, float* D_dev, int64_t* I_dev, int64_t id_offset, void* stream) {
    IVR_TRY(range_args(idx, q_dev, nq, radius, capacity, lims_dev, D_dev, I_dev));
    cudaStream_t st = static_cast<cudaStream_t>(stream);       // NULL = the legacy default stream, as in CUDA
    if (nq == 0) {
        IVR_CUDA(cudaSetDevice(idx->device));
        IVR_CUDA(cudaMemsetAsync(lims_dev, 0, sizeof(int64_t), st));
        return IVR_OK;
    }
    return with_search_window(idx, id_offset, st, "range_search", [&](int64_t id_offset) {
        return range_search_device(idx, q_dev, nq, radius, capacity, lims_dev, D_dev, I_dev, id_offset, st);
    });
}

int ivr_index_range_search_keys_device(ivr_index* idx, const float* q_dev, int64_t nq, float radius, int64_t capacity,
                                       int64_t* lims_dev, uint64_t* keys_dev, int64_t id_offset, void* stream) {
    IVR_TRY(range_args(idx, q_dev, nq, radius, capacity, lims_dev, keys_dev, keys_dev));
    IVR_TRY(check_key_ids(idx, id_offset, "range_search_keys"));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nq == 0) {
        IVR_CUDA(cudaSetDevice(idx->device));
        IVR_CUDA(cudaMemsetAsync(lims_dev, 0, sizeof(int64_t), st));
        return IVR_OK;
    }
    return with_search_window(idx, id_offset, st, "range_search_keys", [&](int64_t id_offset) {
        return range_search_keys_device(idx, q_dev, nq, radius, capacity, lims_dev, keys_dev, id_offset, st);
    });
}

}  // extern "C"

namespace ivr {

// The host-pointer range searches, after their argument checks: queries in, lims and the hits out through the
// handle's pinned and device staging buffers, device_call(q_dev, lims_dev, D_dev, I_dev, stream) in between.
template <class DeviceCall>
static int host_range(ivr_index* idx, const float* q_host, int64_t nq, int64_t capacity, int64_t* lims_host,
                      float* D_host, int64_t* I_host, DeviceCall&& device_call) {
    if (nq == 0) { lims_host[0] = 0; return IVR_OK; }
    IVR_CUDA(cudaSetDevice(idx->device));
    cudaStream_t st = idx->stream;
    const size_t qb = static_cast<size_t>(nq) * idx->dim * sizeof(float);
    const size_t lb = static_cast<size_t>(nq + 1) * sizeof(int64_t);
    const size_t db = static_cast<size_t>(capacity) * sizeof(float), ib = static_cast<size_t>(capacity) * sizeof(int64_t);
    Carve carve;                                                    // the pinned buffer holds the first two parts
    const size_t o_q = carve(qb), o_l = carve(lb);
    IVR_TRY(ensure_pin(idx, carve.size));
    const size_t o_d = carve(db), o_i = carve(ib);
    IVR_TRY(ensure_io(idx, carve.size));
    char* pin = static_cast<char*>(idx->pin);
    char* io = static_cast<char*>(idx->io);
    float* dq = reinterpret_cast<float*>(io + o_q);
    int64_t* dl = reinterpret_cast<int64_t*>(io + o_l);
    float* dd = reinterpret_cast<float*>(io + o_d);
    int64_t* di = reinterpret_cast<int64_t*>(io + o_i);
    memcpy(pin + o_q, q_host, qb);
    IVR_CUDA(cudaMemcpyAsync(dq, pin + o_q, qb, cudaMemcpyHostToDevice, st));
    IVR_TRY(device_call(dq, dl, dd, di, st));
    IVR_CUDA(cudaMemcpyAsync(pin + o_l, dl, lb, cudaMemcpyDeviceToHost, st));
    IVR_CUDA(cudaStreamSynchronize(st));
    memcpy(lims_host, pin + o_l, lb);
    const int64_t total = lims_host[nq];
    if (total == 0 || total > capacity) return IVR_OK;              // nothing to copy / the caller retries
    // the hits, through the pinned buffer sized to what was found
    const size_t hd = static_cast<size_t>(total) * sizeof(float), hi = static_cast<size_t>(total) * sizeof(int64_t);
    Carve hits;
    const size_t o_hd = hits(hd), o_hi = hits(hi);
    IVR_TRY(ensure_pin(idx, hits.size));
    pin = static_cast<char*>(idx->pin);
    IVR_CUDA(cudaMemcpyAsync(pin + o_hd, dd, hd, cudaMemcpyDeviceToHost, st));
    IVR_CUDA(cudaMemcpyAsync(pin + o_hi, di, hi, cudaMemcpyDeviceToHost, st));
    IVR_CUDA(cudaStreamSynchronize(st));
    staged_memcpy(D_host, pin + o_hd, hd);
    staged_memcpy(I_host, pin + o_hi, hi);
    return IVR_OK;
}

}  // namespace ivr

extern "C" {

int ivr_index_range_search(ivr_index* idx, const float* q_host, int64_t nq, float radius, int64_t capacity,
                           int64_t* lims_host, float* D_host, int64_t* I_host) {
    IVR_TRY(range_args(idx, q_host, nq, radius, capacity, lims_host, D_host, I_host));
    return host_range(idx, q_host, nq, capacity, lims_host, D_host, I_host,
                      [&](const float* dq, int64_t* dl, float* dd, int64_t* di, cudaStream_t st) {
        return ivr_index_range_search_device(idx, dq, nq, radius, capacity, dl, dd, di, 0, st);
    });
}

int ivr_index_range_search_selected_device(ivr_index* idx, const ivr_selection* sel, const float* q_dev, int64_t nq,
                                           float radius, int64_t capacity, int64_t* lims_dev, float* D_dev,
                                           int64_t* I_dev, int64_t id_offset, void* stream) {
    IVR_TRY(range_args(idx, q_dev, nq, radius, capacity, lims_dev, D_dev, I_dev));
    IVR_TRY(selected_args(idx, sel, "range_search_selected"));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nq == 0) {
        IVR_CUDA(cudaSetDevice(idx->device));
        IVR_CUDA(cudaMemsetAsync(lims_dev, 0, sizeof(int64_t), st));
        return IVR_OK;
    }
    return with_search_window(idx, id_offset, st, "range_search_selected", [&](int64_t id_offset) {
        return range_search_selected_device(idx, selection_all(sel, idx->ntotal), q_dev, nq, radius, capacity,
                                            lims_dev, D_dev, I_dev, id_offset, st);
    });
}

int ivr_index_search_selected_keys_device(ivr_index* idx, const ivr_selection* sel, const float* q_dev, int64_t nq,
                                          int k, uint64_t* keys_dev, int64_t id_offset, void* stream) {
    if (!idx || nq < 0 || (nq > 0 && (!q_dev || !keys_dev))) {
        set_error("search_selected_keys: bad argument");
        return IVR_EINVAL;
    }
    IVR_TRY(check_key_ids(idx, id_offset, "search_selected_keys"));
    return search_selected_impl(idx, sel, q_dev, nq, k, nullptr, reinterpret_cast<int64_t*>(keys_dev), id_offset,
                                static_cast<cudaStream_t>(stream), "search_selected_keys", /*windowed=*/true);
}

int ivr_index_range_search_selected_keys_device(ivr_index* idx, const ivr_selection* sel, const float* q_dev,
                                                int64_t nq, float radius, int64_t capacity, int64_t* lims_dev,
                                                uint64_t* keys_dev, int64_t id_offset, void* stream) {
    IVR_TRY(range_args(idx, q_dev, nq, radius, capacity, lims_dev, keys_dev, keys_dev));
    IVR_TRY(selected_args(idx, sel, "range_search_selected_keys", /*windowed=*/true));
    IVR_TRY(check_key_ids(idx, id_offset, "range_search_selected_keys"));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nq == 0) {
        IVR_CUDA(cudaSetDevice(idx->device));
        IVR_CUDA(cudaMemsetAsync(lims_dev, 0, sizeof(int64_t), st));
        return IVR_OK;
    }
    return with_selected_window(idx, sel, st, "range_search_selected_keys", [&](const SelCut& cut) {
        return range_search_selected_keys_device(idx, cut, q_dev, nq, radius, capacity, lims_dev, keys_dev, id_offset,
                                                 st);
    });
}

int ivr_index_range_search_selected(ivr_index* idx, const ivr_selection* sel, const float* q_host, int64_t nq,
                                    float radius, int64_t capacity, int64_t* lims_host, float* D_host,
                                    int64_t* I_host) {
    IVR_TRY(range_args(idx, q_host, nq, radius, capacity, lims_host, D_host, I_host));
    IVR_TRY(selected_args(idx, sel, "range_search_selected"));
    return host_range(idx, q_host, nq, capacity, lims_host, D_host, I_host,
                      [&](const float* dq, int64_t* dl, float* dd, int64_t* di, cudaStream_t st) {
        return ivr_index_range_search_selected_device(idx, sel, dq, nq, radius, capacity, dl, dd, di, 0, st);
    });
}

int ivr_index_range_self_join_device(ivr_index* idx, float radius, int64_t capacity, int64_t* lims_dev, float* D_dev,
                                     int64_t* I_dev, void* stream) {
    IVR_TRY(join_args(idx, radius, capacity, lims_dev, D_dev, I_dev));
    cudaStream_t st = static_cast<cudaStream_t>(stream);       // NULL = the legacy default stream, as in CUDA
    return with_search_window(idx, 0, st, "range_self_join", [&](int64_t id_offset) {
        return range_self_join_device(idx, radius, capacity, lims_dev, D_dev, I_dev, id_offset, st);
    });
}

int ivr_index_range_self_join(ivr_index* idx, float radius, int64_t capacity, int64_t* lims_host, float* D_host,
                              int64_t* I_host) {
    IVR_TRY(join_args(idx, radius, capacity, lims_host, D_host, I_host));
    IVR_CUDA(cudaSetDevice(idx->device));
    cudaStream_t st = idx->stream;
    // a window reaching past the rows fails in the device call, before anything is copied back
    const int64_t n = std::min(idx->win_count >= 0 ? idx->win_count : idx->ntotal, idx->ntotal);
    const size_t lb = static_cast<size_t>(n + 1) * sizeof(int64_t);
    const size_t db = static_cast<size_t>(capacity) * sizeof(float), ib = static_cast<size_t>(capacity) * sizeof(int64_t);
    Carve carve;                                                    // the pinned buffer holds the first part
    const size_t o_l = carve(lb);
    IVR_TRY(ensure_pin(idx, carve.size));
    const size_t o_d = carve(db), o_i = carve(ib);
    IVR_TRY(ensure_io(idx, carve.size));
    char* pin = static_cast<char*>(idx->pin);
    char* io = static_cast<char*>(idx->io);
    int64_t* dl = reinterpret_cast<int64_t*>(io + o_l);
    float* dd = reinterpret_cast<float*>(io + o_d);
    int64_t* di = reinterpret_cast<int64_t*>(io + o_i);
    IVR_TRY(ivr_index_range_self_join_device(idx, radius, capacity, dl, dd, di, st));
    IVR_CUDA(cudaMemcpyAsync(pin + o_l, dl, lb, cudaMemcpyDeviceToHost, st));
    IVR_CUDA(cudaStreamSynchronize(st));
    memcpy(lims_host, pin + o_l, lb);
    const int64_t total = lims_host[n];
    if (total == 0 || total > capacity) return IVR_OK;              // nothing to copy / the caller retries
    const size_t hd = static_cast<size_t>(total) * sizeof(float), hi = static_cast<size_t>(total) * sizeof(int64_t);
    Carve hits;
    const size_t o_hd = hits(hd), o_hi = hits(hi);
    IVR_TRY(ensure_pin(idx, hits.size));
    pin = static_cast<char*>(idx->pin);
    IVR_CUDA(cudaMemcpyAsync(pin + o_hd, dd, hd, cudaMemcpyDeviceToHost, st));
    IVR_CUDA(cudaMemcpyAsync(pin + o_hi, di, hi, cudaMemcpyDeviceToHost, st));
    IVR_CUDA(cudaStreamSynchronize(st));
    staged_memcpy(D_host, pin + o_hd, hd);
    staged_memcpy(I_host, pin + o_hi, hi);
    return IVR_OK;
}

int ivr_index_dpad(const ivr_index* idx) { return idx ? idx->dpad : -1; }

int ivr_index_rows_f16_device(ivr_index* idx, int64_t first, int64_t n, void* dst, void* stream) {
    if (!idx || (n > 0 && !dst) || first < 0 || n < 0 || first + n > idx->ntotal) {
        set_error("rows_f16: bad argument (NULL index or dst, or rows [%lld, +%lld) outside the %lld stored rows)",
                  static_cast<long long>(first), static_cast<long long>(n),
                  static_cast<long long>(idx ? idx->ntotal : 0));
        return IVR_EINVAL;
    }
    if (n == 0) return IVR_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    IVR_CUDA(cudaSetDevice(idx->device));
    if (idx->rows_ready_set) IVR_CUDA(cudaStreamWaitEvent(st, idx->rows_ready, 0));   // rows added on another stream
    IVR_CUDA(cudaMemcpyAsync(dst, idx->rows + first * idx->dpad, static_cast<size_t>(n) * idx->dpad * sizeof(__half),
                             cudaMemcpyDeviceToDevice, st));
    return IVR_OK;
}

int ivr_index_range_self_join_keys_device(ivr_index* idx, float radius, int64_t capacity, int64_t* lims_dev,
                                          uint64_t* keys_dev, int64_t id_offset, void* stream) {
    IVR_TRY(join_args(idx, radius, capacity, lims_dev, keys_dev, keys_dev));
    IVR_TRY(check_key_ids(idx, id_offset, "range_self_join_keys"));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return with_search_window(idx, id_offset, st, "range_self_join_keys", [&](int64_t id_offset) {
        return range_self_join_keys_device(idx, radius, capacity, lims_dev, keys_dev, id_offset, st);
    });
}

int ivr_index_range_cross_join_keys_device(ivr_index* idx, const void* other_rows, int64_t n_other,
                                           int64_t other_first_id, int other_is_lower, float radius,
                                           int64_t capacity, int64_t* lims_dev, uint64_t* keys_dev,
                                           int64_t id_offset, void* stream) {
    if (radius != radius) { set_error("range_cross_join: radius is NaN"); return IVR_EINVAL; }
    if (capacity < 0 || n_other < 0) {
        set_error("range_cross_join: capacity and n_other must be >= 0 (got %lld, %lld)",
                  static_cast<long long>(capacity), static_cast<long long>(n_other));
        return IVR_EINVAL;
    }
    if (!idx || !lims_dev || (capacity > 0 && !keys_dev) || (n_other > 0 && !other_rows)) {
        set_error("range_cross_join: bad argument (NULL index or buffer)");
        return IVR_EINVAL;
    }
    if (capacity > INT_MAX) {
        set_error("range_cross_join: at most 2^31-1 hits per call (capacity %lld)", static_cast<long long>(capacity));
        return IVR_EUNSUPPORTED;
    }
    if (small_range_chunk(idx) < 16) {
        set_error("range_cross_join: dim %d is wider than the small-batch kernel holds (padded dim <= 4096)", idx->dim);
        return IVR_EUNSUPPORTED;
    }
    const int64_t n_self = idx->win_count >= 0 ? idx->win_count : idx->ntotal;
    if (n_self + n_other >= INT_MAX) {
        set_error("range_cross_join: at most 2^31-2 rows on both sides together (%lld + %lld)",
                  static_cast<long long>(n_self), static_cast<long long>(n_other));
        return IVR_EUNSUPPORTED;
    }
    IVR_TRY(check_key_ids(idx, id_offset, "range_cross_join"));
    if (other_first_id < 0 || other_first_id + n_other > 0x100000000ll) {
        set_error("range_cross_join: global row ids must stay below 2^32 (other rows %lld + %lld)",
                  static_cast<long long>(other_first_id), static_cast<long long>(n_other));
        return IVR_EUNSUPPORTED;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return with_search_window(idx, id_offset, st, "range_cross_join", [&](int64_t id_offset) {
        return range_cross_join_keys_device(idx, static_cast<const __half*>(other_rows), n_other, other_is_lower != 0,
                                            static_cast<uint32_t>(id_offset), static_cast<uint32_t>(other_first_id),
                                            radius, capacity, lims_dev, keys_dev, st);
    });
}

int ivr_index_set_timing(ivr_index* idx, int enable) {
    if (!idx) { set_error("NULL index"); return IVR_EINVAL; }
    idx->timing = enable != 0;
    return IVR_OK;
}

int ivr_index_last_timing(ivr_index* idx, float ms[3], int launches[3]) {
    if (!idx || !ms) { set_error("last_timing: bad argument"); return IVR_EINVAL; }
    IVR_CUDA(cudaSetDevice(idx->device));
    for (int i = 0; i < 3; ++i) {
        ms[i] = 0.f;
        if (idx->ev_valid[i]) {
            IVR_CUDA(cudaEventSynchronize(idx->ev[2 * i + 1]));
            IVR_CUDA(cudaEventElapsedTime(&ms[i], idx->ev[2 * i], idx->ev[2 * i + 1]));
        }
        if (launches) launches[i] = idx->launches[i];
    }
    return IVR_OK;
}

int ivr_index_last_path(const ivr_index* idx) { return idx ? idx->last_path : -1; }
const char* ivr_index_last_kernel(const ivr_index* idx) { return idx ? idx->last_kernel : ""; }

int ivr_topk_merge_device(int device, const float* D_parts, const int64_t* I_parts, int n_parts,
                          int64_t nq, int k, float* D_out, int64_t* I_out, void* stream) {
    if (n_parts <= 0 || nq < 0 || k <= 0 || !D_parts || !I_parts || !D_out || !I_out) {
        set_error("topk_merge: bad argument");
        return IVR_EINVAL;
    }
    if (k > IVR_MAX_K) { set_error("topk_merge: k=%d exceeds IVR_MAX_K", k); return IVR_EUNSUPPORTED; }
    if (nq == 0) return IVR_OK;
    IVR_TRY(require_device(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t n = static_cast<int64_t>(n_parts) * nq * k;
    const size_t tmp_keys = merge_tmp_entries(n_parts, nq, k);
    uint64_t* keys = nullptr;
    IVR_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&keys), (n + tmp_keys) * sizeof(uint64_t) +
                             (static_cast<size_t>(n_parts) * nq + 64) * sizeof(int), st));
    int rc = pack_parts(D_parts, I_parts, keys, n, st);
    if (rc == IVR_OK) {
        MergeIn in{};
        in.entries = keys; in.counts = nullptr;
        in.list_stride = nq * k; in.q_stride = k;
        in.n_lists = n_parts; in.fixed_count = k;
        rc = merge_lists_final(in, nq, k, D_out, I_out, 0, keys + n,
                               reinterpret_cast<int*>(keys + n + tmp_keys), st, nullptr);
    }
    cudaFreeAsync(keys, st);
    return rc;
}

int ivr_topk_merge_keys_device(int device, const uint64_t* keys_parts, int n_parts, int64_t nq, int k,
                               float* D_out, int64_t* I_out, void* stream) {
    if (n_parts <= 0 || nq < 0 || k <= 0 || !keys_parts || !D_out || !I_out) {
        set_error("topk_merge_keys: bad argument");
        return IVR_EINVAL;
    }
    if (k > IVR_MAX_K) { set_error("topk_merge_keys: k=%d exceeds IVR_MAX_K", k); return IVR_EUNSUPPORTED; }
    if (merge_tmp_entries(n_parts, nq, k) != 0) {     // one merge level needs no scratch: no allocation on this path
        set_error("topk_merge_keys: at most 64 parts (got %d)", n_parts);
        return IVR_EUNSUPPORTED;
    }
    if (nq == 0) return IVR_OK;
    IVR_TRY(require_device_once(device));
    MergeIn in{};
    in.entries = keys_parts; in.counts = nullptr;
    in.list_stride = nq * k; in.q_stride = k;
    in.n_lists = n_parts; in.fixed_count = k;
    return merge_lists_final(in, nq, k, D_out, I_out, 0, nullptr, nullptr, static_cast<cudaStream_t>(stream), nullptr);
}

int ivr_range_merge_keys_device(int device, const uint64_t* keys_parts, int64_t part_stride, const int64_t* lims_parts,
                                int n_parts, int64_t nq, int64_t* lims, float* D, int64_t* I, void* stream) {
    if (n_parts < 1 || n_parts > 64 || nq < 0 || part_stride < 0 || !lims_parts || !lims ||
        (part_stride > 0 && (!keys_parts || !D || !I))) {
        set_error("range_merge_keys: bad argument (n_parts %d of 1..64, nq %lld, part_stride %lld, or a NULL buffer)",
                  n_parts, static_cast<long long>(nq), static_cast<long long>(part_stride));
        return IVR_EINVAL;
    }
    if (part_stride > INT64_MAX / n_parts || nq >= INT64_MAX / 64) {
        set_error("range_merge_keys: n_parts * part_stride or n_parts * (nq + 1) overflows");
        return IVR_EINVAL;
    }
    IVR_TRY(require_device_once(device));
    return range_merge_keys_device(keys_parts, part_stride, lims_parts, n_parts, nq, lims, D, I,
                                   static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------ normalise ----
int ivr_normalize_l2_device(int device, float* x_dev, int64_t n, int d, void* stream) {
    if (n < 0 || d <= 0 || (n > 0 && !x_dev)) { set_error("normalize_l2: bad argument"); return IVR_EINVAL; }
    IVR_TRY(require_device(device));
    return normalize_l2_device(x_dev, n, d, static_cast<cudaStream_t>(stream));
}

int ivr_normalize_l2(int device, float* x_host, int64_t n, int d) {
    if (n < 0 || d <= 0 || (n > 0 && !x_host)) { set_error("normalize_l2: bad argument"); return IVR_EINVAL; }
    if (n == 0) return IVR_OK;
    IVR_TRY(require_device(device));
    const size_t bytes = static_cast<size_t>(n) * d * sizeof(float);
    DevBuf b;
    IVR_TRY(b.alloc(bytes));
    IVR_CUDA(cudaMemcpy(b.p, x_host, bytes, cudaMemcpyHostToDevice));
    IVR_TRY(normalize_l2_device(static_cast<float*>(b.p), n, d, nullptr));
    IVR_CUDA(cudaMemcpy(x_host, b.p, bytes, cudaMemcpyDeviceToHost));
    return IVR_OK;
}

// ---------------------------------------------------------------- dedup ----
int ivr_dedup_set_timing(int enable) { return dedup_set_timing(enable); }
int ivr_dedup_last_timing(float ms[2]) { return ms ? dedup_last_timing(ms) : IVR_EINVAL; }

int ivr_consecutive_cosine_device(int device, const float* e_dev, int64_t n, int d, float* out_dev,
                                  void* stream) {
    // out_dev: n floats, out[i] = cos(e_i, e_{i-1}), out[0] = 1  (device variant keeps the
    // frame-aligned layout; the host variant below drops element 0 like the reference list)
    if (n < 0 || d <= 0 || (n > 0 && (!e_dev || !out_dev))) { set_error("consecutive_cosine: bad argument"); return IVR_EINVAL; }
    if (n == 0) return IVR_OK;
    IVR_TRY(require_device(device));
    int sm = 0;
    IVR_CUDA(cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device));
    return launch_banded(e_dev, n, 0, d, 1, 2.0f, nullptr, out_dev, sm, static_cast<cudaStream_t>(stream));
}

int ivr_consecutive_cosine(int device, const float* e_host, int64_t n, int d, float* out_host) {
    if (n < 0 || d <= 0 || (n > 0 && !e_host) || (n > 1 && !out_host)) { set_error("consecutive_cosine: bad argument"); return IVR_EINVAL; }
    if (n <= 1) return IVR_OK;
    IVR_TRY(require_device(device));
    const size_t bytes = static_cast<size_t>(n) * d * sizeof(float);
    DevBuf e, o;
    IVR_TRY(e.alloc(bytes)); IVR_TRY(o.alloc(n * sizeof(float)));
    IVR_CUDA(cudaMemcpy(e.p, e_host, bytes, cudaMemcpyHostToDevice));
    IVR_TRY(ivr_consecutive_cosine_device(device, static_cast<float*>(e.p), n, d, static_cast<float*>(o.p), nullptr));
    IVR_CUDA(cudaMemcpy(out_host, static_cast<float*>(o.p) + 1, (n - 1) * sizeof(float), cudaMemcpyDeviceToHost));
    return IVR_OK;
}

int ivr_dedup_window_device(int device, const float* e_dev, int64_t n, int d,
                            const int64_t* scene_start_dev, const int64_t* scene_end_dev,
                            int64_t n_scenes, int window, float thr, uint8_t* keep_dev,
                            float* cos_prev_dev, uint32_t* mask_ws_dev, void* stream) {
    if (n < 0 || d <= 0 || n_scenes < 0 || (n > 0 && (!e_dev || !keep_dev || !mask_ws_dev)) ||
        (n_scenes > 0 && (!scene_start_dev || !scene_end_dev))) {
        set_error("dedup_window: bad argument");
        return IVR_EINVAL;
    }
    if (window < 1 || window > IVR_MAX_WINDOW) {
        set_error("dedup_window: window %d outside 1..%d", window, IVR_MAX_WINDOW);
        return IVR_EUNSUPPORTED;
    }
    if (n == 0) return IVR_OK;
    IVR_TRY(require_device(device));
    return dedup_window_device(device, e_dev, n, d, scene_start_dev, scene_end_dev, n_scenes, window,
                               thr, keep_dev, cos_prev_dev, mask_ws_dev, static_cast<cudaStream_t>(stream));
}

int ivr_frame_filter(int device, const float* e_host, int64_t n, int d, int window, float thr, float transition_thr,
                     int min_scene_len, uint8_t* keep_host, float* cos_prev_host, int64_t* stats) {
    if (n < 0 || d <= 0 || (n > 0 && (!e_host || !keep_host))) { set_error("frame_filter: bad argument"); return IVR_EINVAL; }
    if (window > IVR_MAX_WINDOW) {
        set_error("frame_filter: window %d above %d", window, IVR_MAX_WINDOW);
        return IVR_EUNSUPPORTED;
    }
    if (stats) stats[0] = stats[1] = 0;
    if (n == 0) return IVR_OK;
    IVR_TRY(require_device(device));
    int sm = 0;
    IVR_CUDA(cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device));
    static thread_local cudaStream_t st = nullptr;
    static thread_local int st_device = -1;
    if (st_device != device) {
        if (st) cudaStreamDestroy(st);
        IVR_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        st_device = device;
    }
    const int w_kernel = window < 1 ? 1 : window;                     // masks of an empty window are never consulted
    const int halo = w_kernel;
    const size_t row_bytes = static_cast<size_t>(d) * sizeof(float);
    int64_t chunk = std::max<int64_t>(halo + 1, (static_cast<int64_t>(64) << 20) / static_cast<int64_t>(row_bytes));
    chunk = std::min(chunk, n);
    // Is the caller's buffer page-locked?  Then the chunks are copied straight from it; otherwise they are staged
    // through two pinned buffers filled by a few host threads while the previous chunk is on the wire.
    cudaPointerAttributes attr{};
    const bool pinned = cudaPointerGetAttributes(&attr, e_host) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    DevBuf buf, masks, cosp, keep, cnt;
    IVR_TRY(buf.alloc((chunk + halo) * row_bytes, st));
    IVR_TRY(masks.alloc(n * sizeof(uint32_t), st)); IVR_TRY(cosp.alloc(n * sizeof(float), st));
    IVR_TRY(keep.alloc(n, st)); IVR_TRY(cnt.alloc(16, st));
    void* pin = nullptr;
    cudaEvent_t done[2] = {nullptr, nullptr};
    int rc = IVR_OK;
    if (!pinned) {
        static thread_local void* tl_pin = nullptr;
        static thread_local size_t tl_pin_bytes = 0;
        if (tl_pin_bytes < 2 * chunk * row_bytes) {
            if (tl_pin) cudaFreeHost(tl_pin);
            tl_pin = nullptr; tl_pin_bytes = 0;
            IVR_CUDA(cudaMallocHost(&tl_pin, 2 * chunk * row_bytes));
            tl_pin_bytes = 2 * chunk * row_bytes;
        }
        pin = tl_pin;
        for (auto& e : done) IVR_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    float* dbuf = static_cast<float*>(buf.p);
    IVR_CUDA(cudaMemsetAsync(cnt.p, 0, 16, st));
    int64_t off = 0;
    for (int it = 0; off < n && rc == IVR_OK; ++it) {
        const int64_t m = std::min(chunk, n - off);
        const int64_t ctx = std::min<int64_t>(halo, off);             // look-back frames kept from the previous chunk
        const float* src = e_host + off * d;
        if (!pinned) {
            const int b = it & 1;
            char* p = static_cast<char*>(pin) + b * chunk * row_bytes;
            if (it >= 2 && cudaEventSynchronize(done[b]) != cudaSuccess) { rc = IVR_ECUDA; break; }
            staged_memcpy(p, src, m * row_bytes);
            src = reinterpret_cast<const float*>(p);
        }
        if (cudaMemcpyAsync(dbuf + halo * d, src, m * row_bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) { rc = IVR_ECUDA; break; }
        if (!pinned) cudaEventRecord(done[it & 1], st);
        // buffer rows [halo - ctx, halo + m) hold frames [off - ctx, off + m); outputs go to frames [off, off + m)
        rc = launch_banded(dbuf + (halo - ctx) * d, ctx + m, ctx, d, w_kernel, thr,
                           static_cast<uint32_t*>(masks.p) + (off - ctx), static_cast<float*>(cosp.p) + (off - ctx), sm, st);
        if (rc != IVR_OK) break;
        if (off + m < n &&                                            // keep the last `halo` frames as the next chunk's context
            cudaMemcpyAsync(dbuf + std::max<int64_t>(0, halo - m) * d, dbuf + std::max<int64_t>(halo, m) * d,
                            std::min<int64_t>(halo, m) * row_bytes, cudaMemcpyDeviceToDevice, st) != cudaSuccess) { rc = IVR_ECUDA; break; }
        off += m;
    }
    if (rc == IVR_OK)
        rc = launch_scene_resolve(static_cast<uint32_t*>(masks.p), static_cast<float*>(cosp.p), n, window, transition_thr,
                                  min_scene_len, static_cast<uint8_t*>(keep.p), static_cast<unsigned long long*>(cnt.p), st);
    unsigned long long scenes[2] = {0, 0};
    if (rc == IVR_OK) {
        cudaMemcpyAsync(keep_host, keep.p, n, cudaMemcpyDeviceToHost, st);
        if (cos_prev_host) cudaMemcpyAsync(cos_prev_host, cosp.p, n * sizeof(float), cudaMemcpyDeviceToHost, st);
        cudaMemcpyAsync(scenes, cnt.p, 16, cudaMemcpyDeviceToHost, st);
    }
    const cudaError_t e = cudaStreamSynchronize(st);
    for (auto& ev : done) if (ev) cudaEventDestroy(ev);
    if (rc == IVR_OK && e != cudaSuccess) { set_error("frame_filter: %s", cudaGetErrorString(e)); rc = IVR_ECUDA; }
    if (rc == IVR_ECUDA && g_err[0] == 0) set_error("frame_filter: CUDA failure");
    if (rc == IVR_OK && stats) { stats[0] = static_cast<int64_t>(scenes[0]); stats[1] = static_cast<int64_t>(scenes[1]); }
    return rc;
}

int ivr_dedup_window(int device, const float* e_host, int64_t n, int d, const int64_t* scene_start,
                     const int64_t* scene_end, int64_t n_scenes, int window, float thr,
                     uint8_t* keep_host, float* cos_prev_host) {
    if (n < 0 || d <= 0 || n_scenes < 0 || (n > 0 && (!e_host || !keep_host)) ||
        (n_scenes > 0 && (!scene_start || !scene_end))) {
        set_error("dedup_window: bad argument");
        return IVR_EINVAL;
    }
    if (window < 1 || window > IVR_MAX_WINDOW) {
        set_error("dedup_window: window %d outside 1..%d", window, IVR_MAX_WINDOW);
        return IVR_EUNSUPPORTED;
    }
    if (n == 0) return IVR_OK;
    IVR_TRY(require_device(device));
    const size_t bytes = static_cast<size_t>(n) * d * sizeof(float);
    DevBuf e, m, c, k, ss, se;
    IVR_TRY(e.alloc(bytes)); IVR_TRY(m.alloc(n * sizeof(uint32_t))); IVR_TRY(c.alloc(n * sizeof(float)));
    IVR_TRY(k.alloc(n)); IVR_TRY(ss.alloc(n_scenes * sizeof(int64_t))); IVR_TRY(se.alloc(n_scenes * sizeof(int64_t)));
    IVR_CUDA(cudaMemcpy(e.p, e_host, bytes, cudaMemcpyHostToDevice));
    if (n_scenes > 0) {
        IVR_CUDA(cudaMemcpy(ss.p, scene_start, n_scenes * sizeof(int64_t), cudaMemcpyHostToDevice));
        IVR_CUDA(cudaMemcpy(se.p, scene_end, n_scenes * sizeof(int64_t), cudaMemcpyHostToDevice));
    }
    IVR_TRY(dedup_window_device(device, static_cast<float*>(e.p), n, d, static_cast<int64_t*>(ss.p),
                                static_cast<int64_t*>(se.p), n_scenes, window, thr,
                                static_cast<uint8_t*>(k.p), static_cast<float*>(c.p),
                                static_cast<uint32_t*>(m.p), nullptr));
    IVR_CUDA(cudaMemcpy(keep_host, k.p, n, cudaMemcpyDeviceToHost));
    if (cos_prev_host) IVR_CUDA(cudaMemcpy(cos_prev_host, c.p, n * sizeof(float), cudaMemcpyDeviceToHost));
    return IVR_OK;
}

static int dedup_chain_host(int device, const float* e_host, int64_t n, int d, const int64_t* scene_start,
                           const int64_t* scene_end, int64_t n_scenes, int min_distance, float thr,
                           int force_last, int fifo, uint8_t* keep_host, const char* who) {
    if (n < 0 || d <= 0 || n_scenes < 0 || (n > 0 && (!e_host || !keep_host)) ||
        (n_scenes > 0 && (!scene_start || !scene_end))) {
        set_error("%s: bad argument", who);
        return IVR_EINVAL;
    }
    if (fifo < 1 || fifo > 16) { set_error("%s: fifo %d outside 1..16", who, fifo); return IVR_EUNSUPPORTED; }
    if (n == 0) return IVR_OK;
    IVR_TRY(require_device(device));
    const size_t bytes = static_cast<size_t>(n) * d * sizeof(float);
    DevBuf e, k, ss, se;
    IVR_TRY(e.alloc(bytes)); IVR_TRY(k.alloc(n));
    IVR_TRY(ss.alloc(n_scenes * sizeof(int64_t))); IVR_TRY(se.alloc(n_scenes * sizeof(int64_t)));
    IVR_CUDA(cudaMemcpy(e.p, e_host, bytes, cudaMemcpyHostToDevice));
    if (n_scenes > 0) {
        IVR_CUDA(cudaMemcpy(ss.p, scene_start, n_scenes * sizeof(int64_t), cudaMemcpyHostToDevice));
        IVR_CUDA(cudaMemcpy(se.p, scene_end, n_scenes * sizeof(int64_t), cudaMemcpyHostToDevice));
    }
    IVR_TRY(dedup_chain_device(static_cast<float*>(e.p), n, d, static_cast<int64_t*>(ss.p),
                               static_cast<int64_t*>(se.p), n_scenes, min_distance, thr, force_last, fifo,
                               static_cast<uint8_t*>(k.p), nullptr));
    IVR_CUDA(cudaMemcpy(keep_host, k.p, n, cudaMemcpyDeviceToHost));
    return IVR_OK;
}

int ivr_dedup_chain(int device, const float* e_host, int64_t n, int d, const int64_t* scene_start,
                    const int64_t* scene_end, int64_t n_scenes, int min_distance, float thr,
                    int force_last, uint8_t* keep_host) {
    return dedup_chain_host(device, e_host, n, d, scene_start, scene_end, n_scenes, min_distance, thr,
                            force_last, 1, keep_host, "dedup_chain");
}

int ivr_dedup_fifo(int device, const float* e_host, int64_t n, int d, const int64_t* scene_start,
                   const int64_t* scene_end, int64_t n_scenes, int fifo, float thr, uint8_t* keep_host) {
    return dedup_chain_host(device, e_host, n, d, scene_start, scene_end, n_scenes, 1, thr, 0, fifo, keep_host,
                            "dedup_fifo");
}

int ivr_sequence_similarity(int device, const float* target_host, int64_t nt, const float* db_host, int64_t nd,
                            int dim, int seq_len, float threshold, int64_t max_hits, int32_t* hit_t, int64_t* hit_j,
                            float* hit_sim, int64_t* n_hits) {
    if (nt < 0 || nd < 0 || dim <= 0 || max_hits < 0 || !n_hits || (nt > 0 && !target_host) || (nd > 0 && !db_host) ||
        (max_hits > 0 && (!hit_t || !hit_j || !hit_sim))) {
        set_error("sequence_similarity: bad argument");
        return IVR_EINVAL;
    }
    if (seq_len < 1 || seq_len > IVR_MAX_SEQ_LEN) {
        set_error("sequence_similarity: seq_len %d outside 1..%d", seq_len, IVR_MAX_SEQ_LEN);
        return IVR_EUNSUPPORTED;
    }
    if (nt - seq_len + 1 > 65535) {                                // one grid row per target window start
        set_error("sequence_similarity: more than 65535 target windows (nt=%lld)", static_cast<long long>(nt));
        return IVR_EUNSUPPORTED;
    }
    *n_hits = 0;
    if (nt < seq_len || nd < seq_len) return IVR_OK;
    IVR_TRY(require_device(device));
    const int64_t cols = sequence_block_cols(nt, nd, seq_len);
    DevBuf t, d, tn, dn, cb, ht, hj, hs, cnt;
    IVR_TRY(t.alloc(static_cast<size_t>(nt) * dim * 4)); IVR_TRY(d.alloc(static_cast<size_t>(nd) * dim * 4));
    IVR_TRY(tn.alloc(static_cast<size_t>(nt) * dim * 4)); IVR_TRY(dn.alloc(static_cast<size_t>(nd) * dim * 4));
    IVR_TRY(cb.alloc(static_cast<size_t>(nt) * cols * 4));
    IVR_TRY(ht.alloc(std::max<size_t>(max_hits, 1) * 4)); IVR_TRY(hj.alloc(std::max<size_t>(max_hits, 1) * 8));
    IVR_TRY(hs.alloc(std::max<size_t>(max_hits, 1) * 4)); IVR_TRY(cnt.alloc(8));
    IVR_CUDA(cudaMemcpy(t.p, target_host, static_cast<size_t>(nt) * dim * 4, cudaMemcpyHostToDevice));
    IVR_CUDA(cudaMemcpy(d.p, db_host, static_cast<size_t>(nd) * dim * 4, cudaMemcpyHostToDevice));
    IVR_CUDA(cudaMemset(cnt.p, 0, 8));
    IVR_TRY(sequence_similarity_device(static_cast<float*>(t.p), nt, static_cast<float*>(d.p), nd, dim, seq_len,
                                       threshold, max_hits, static_cast<int32_t*>(ht.p), static_cast<int64_t*>(hj.p),
                                       static_cast<float*>(hs.p), static_cast<unsigned long long*>(cnt.p),
                                       static_cast<float*>(tn.p), static_cast<float*>(dn.p), static_cast<float*>(cb.p),
                                       cols, nullptr));
    unsigned long long total = 0;
    IVR_CUDA(cudaMemcpy(&total, cnt.p, 8, cudaMemcpyDeviceToHost));
    *n_hits = static_cast<int64_t>(total);
    const size_t stored = static_cast<size_t>(std::min<unsigned long long>(total, static_cast<unsigned long long>(max_hits)));
    if (stored) {
        IVR_CUDA(cudaMemcpy(hit_t, ht.p, stored * 4, cudaMemcpyDeviceToHost));
        IVR_CUDA(cudaMemcpy(hit_j, hj.p, stored * 8, cudaMemcpyDeviceToHost));
        IVR_CUDA(cudaMemcpy(hit_sim, hs.p, stored * 4, cudaMemcpyDeviceToHost));
    }
    return IVR_OK;
}

int ivr_cosine_neighbors(int device, const float* e_host, int64_t n, int dim, float eps, uint32_t* adj_host) {
    if (n < 0 || dim <= 0 || (n > 0 && (!e_host || !adj_host))) { set_error("cosine_neighbors: bad argument"); return IVR_EINVAL; }
    if (n > IVR_MAX_CLUSTER_FRAMES) {
        set_error("cosine_neighbors: %lld frames exceed IVR_MAX_CLUSTER_FRAMES=%d", static_cast<long long>(n), IVR_MAX_CLUSTER_FRAMES);
        return IVR_EUNSUPPORTED;
    }
    if (n == 0) return IVR_OK;
    IVR_TRY(require_device(device));
    const size_t words = static_cast<size_t>((n + 31) / 32);
    DevBuf e, xn, cm, adj;
    IVR_TRY(e.alloc(static_cast<size_t>(n) * dim * 4)); IVR_TRY(xn.alloc(static_cast<size_t>(n) * dim * 4));
    IVR_TRY(cm.alloc(static_cast<size_t>(n) * n * 4)); IVR_TRY(adj.alloc(static_cast<size_t>(n) * words * 4));
    IVR_CUDA(cudaMemcpy(e.p, e_host, static_cast<size_t>(n) * dim * 4, cudaMemcpyHostToDevice));
    IVR_TRY(cosine_neighbors_device(static_cast<float*>(e.p), static_cast<int>(n), dim, eps, static_cast<float*>(xn.p),
                                    static_cast<float*>(cm.p), static_cast<uint32_t*>(adj.p), nullptr));
    IVR_CUDA(cudaMemcpy(adj_host, adj.p, static_cast<size_t>(n) * words * 4, cudaMemcpyDeviceToHost));
    return IVR_OK;
}

}  // extern "C"

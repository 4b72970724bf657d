// index.cu -- storage side of the flat inner-product index.
//
// Replaces faiss.IndexFlatIP(d) / .add / .reset / .ntotal and faiss.normalize_L2
// (unified_index.py:1767-1779; core.py:1208, 827).  Rows live in HBM as fp16,
// row-major, the dimension padded to a multiple of 64 so that every row is a
// whole number of 128-byte TMA/UMMA swizzle atoms; ids are the insertion order.
#include "index.cuh"

#include <algorithm>
#include <cstring>

namespace ivr {

int ensure_ws(ivr_index* idx, size_t bytes) {
    if (bytes <= idx->ws_bytes) return IVR_OK;
    IVR_CUDA(cudaSetDevice(idx->device));
    if (idx->ws) {
        // the old buffer may still be in use by work queued on any stream
        IVR_CUDA(cudaDeviceSynchronize());
        IVR_CUDA(cudaFree(idx->ws));
        idx->ws = nullptr; idx->ws_bytes = 0;
    }
    const size_t want = std::max(bytes + bytes / 4, static_cast<size_t>(1) << 20);
    IVR_CUDA(cudaMalloc(&idx->ws, want));
    idx->ws_bytes = want;
    return IVR_OK;
}

int ensure_io(ivr_index* idx, size_t bytes) {
    if (bytes <= idx->io_bytes) return IVR_OK;
    IVR_CUDA(cudaSetDevice(idx->device));
    if (idx->io) {
        IVR_CUDA(cudaDeviceSynchronize());
        IVR_CUDA(cudaFree(idx->io));
        idx->io = nullptr; idx->io_bytes = 0;
    }
    IVR_CUDA(cudaMalloc(&idx->io, bytes));
    idx->io_bytes = bytes;
    return IVR_OK;
}

int ensure_pin(ivr_index* idx, size_t bytes) {
    if (bytes <= idx->pin_bytes) return IVR_OK;
    IVR_CUDA(cudaSetDevice(idx->device));
    if (idx->pin) {
        IVR_CUDA(cudaStreamSynchronize(idx->stream));
        IVR_CUDA(cudaFreeHost(idx->pin));
        idx->pin = nullptr; idx->pin_bytes = 0;
    }
    IVR_CUDA(cudaMallocHost(&idx->pin, bytes));
    idx->pin_bytes = bytes;
    return IVR_OK;
}

int ensure_capacity(ivr_index* idx, int64_t rows, cudaStream_t st, bool exact) {
    if (rows <= idx->capacity) return IVR_OK;
    IVR_CUDA(cudaSetDevice(idx->device));
    int64_t cap = exact ? rows : std::max<int64_t>(rows, idx->capacity + idx->capacity / 2);
    cap = std::max<int64_t>(cap, 1024);
    __half* nr = nullptr;
    const size_t row_bytes = static_cast<size_t>(idx->dpad) * sizeof(__half);
    cudaError_t e = cudaMalloc(&nr, static_cast<size_t>(cap) * row_bytes);
    if (e != cudaSuccess && cap > rows) {          // retry with the exact size
        cudaGetLastError();
        cap = rows;
        e = cudaMalloc(&nr, static_cast<size_t>(cap) * row_bytes);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("cannot allocate %lld rows x %d fp16 on device %d: %s",
                  static_cast<long long>(cap), idx->dpad, idx->device, cudaGetErrorString(e));
        return IVR_ENOMEM;
    }
    if (idx->rows) {
        // Earlier adds may have queued their fp32 -> fp16 conversion on OTHER streams (add_device runs on the
        // caller's stream) and searches may still read the old block: drain the device before the copy, so the
        // copy sees every row and nobody touches the block after it is freed.
        IVR_CUDA(cudaDeviceSynchronize());
        if (idx->ntotal > 0)
            IVR_CUDA(cudaMemcpyAsync(nr, idx->rows, static_cast<size_t>(idx->ntotal) * row_bytes,
                                     cudaMemcpyDeviceToDevice, st));
        IVR_CUDA(cudaStreamSynchronize(st));
        IVR_CUDA(cudaFree(idx->rows));
    }
    idx->rows = nr;
    idx->capacity = cap;
    idx->tmap_rows_n = -1;                           // TMA descriptor is stale
    return IVR_OK;
}

// fp32 [n, dim] -> fp16 [n, dpad] (round-to-nearest-even, saturating at +-65504, zero padded).  NaN stays NaN:
// such a row scores NaN against every query, and the searches never return a NaN score.
// The reference only ever adds L2-normalised rows (unified_index.py:1776, core.py:1189-1196), for
// which fp16 (11 significant bits) is 8x more accurate than bf16 at the same tensor-core rate.
__global__ void rows_to_f16_kernel(const float* __restrict__ src, __half* __restrict__ dst,
                                   int64_t n, int dim, int dpad) {
    const int64_t total = n * (dpad / 2);
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t r = i / (dpad / 2);
        const int c = static_cast<int>(i % (dpad / 2)) * 2;
        float a = (c < dim) ? src[r * dim + c] : 0.f;
        float b = (c + 1 < dim) ? src[r * dim + c + 1] : 0.f;
        if (!isnan(a)) a = fminf(fmaxf(a, -65504.f), 65504.f);
        if (!isnan(b)) b = fminf(fmaxf(b, -65504.f), 65504.f);
        reinterpret_cast<__half2*>(dst)[i] = __floats2half2_rn(a, b);
    }
}

int convert_rows(ivr_index* idx, const float* src_dev, int64_t n, int64_t dst_row, cudaStream_t st) {
    if (n <= 0) return IVR_OK;
    const int64_t total = n * (idx->dpad / 2);
    const int threads = 256;
    const int64_t blocks = std::min<int64_t>((total + threads - 1) / threads,
                                             static_cast<int64_t>(idx->sm_count) * 16);
    rows_to_f16_kernel<<<static_cast<unsigned>(blocks), threads, 0, st>>>(
        src_dev, idx->rows + dst_row * idx->dpad, n, idx->dim, idx->dpad);
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

// fp16 [n, dpad] rows -> fp32 [n, dim] (exact widening; the padding columns are dropped)
__global__ void rows_to_f32_kernel(const __half* __restrict__ src, float* __restrict__ dst, int64_t n, int dim, int dpad) {
    const int64_t total = n * dim;
    for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t r = i / dim;
        const int c = static_cast<int>(i % dim);
        dst[i] = __half2float(src[r * dpad + c]);
    }
}

int reconstruct_rows(ivr_index* idx, int64_t first, int64_t n, float* dst_dev, cudaStream_t st) {
    if (n <= 0) return IVR_OK;
    const int64_t total = n * idx->dim;
    const int threads = 256;
    const int64_t blocks = std::min<int64_t>((total + threads - 1) / threads, static_cast<int64_t>(idx->sm_count) * 16);
    rows_to_f32_kernel<<<static_cast<unsigned>(blocks), threads, 0, st>>>(idx->rows + first * idx->dpad, dst_dev, n,
                                                                          idx->dim, idx->dpad);
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

// In-place row L2 normalisation; one warp per row; zero rows untouched
// (faiss.normalize_L2 / fvec_renorm_L2 semantics).
__global__ void normalize_l2_kernel(float* __restrict__ x, int64_t n, int d) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
    if (row >= n) return;
    float* p = x + row * d;
    float ss = 0.f;
    for (int c = lane; c < d; c += 32) { const float v = p[c]; ss = fmaf(v, v, ss); }
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if (ss > 0.f) {
        const float inv = 1.0f / sqrtf(ss);
        for (int c = lane; c < d; c += 32) p[c] *= inv;
    }
}

int normalize_l2_device(float* x_dev, int64_t n, int d, cudaStream_t st) {
    if (n <= 0 || d <= 0) return IVR_OK;
    const int threads = 256;
    const int64_t blocks = (n * 32 + threads - 1) / threads;
    normalize_l2_kernel<<<static_cast<unsigned>(blocks), threads, 0, st>>>(x_dev, n, d);
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

}  // namespace ivr

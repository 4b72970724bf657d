// search_stream.cu -- K3: bandwidth-bound small-batch exact search.
//
// Replaces index.search(x, k) for nq <= 4 per pass (the reference's production
// call is nq = 1: unified_index.py:503).  The fp16 row matrix is streamed once
// with 128-bit coalesced, L1-bypassing loads; every 8 lanes own one row, so a
// warp covers 4 rows per step and keeps 2 steps (8 rows) of loads in flight.
// The 8-row groups are dealt to the warps ROUND-ROBIN (group g -> warp g mod W):
// at any moment the grid reads one contiguous window of the matrix, and -- what
// the merge relies on -- neighbouring rows (near-duplicate frames of one video)
// end up in different warps' lists.
// Scores are reduced with 3 shuffles and go straight into a per-warp candidate
// list guarded by a running admission threshold (the warp's current k-th best);
// full lists are compacted in registers (warp bitonic sort).  No score ever
// reaches HBM.  Every warp also publishes the MAXIMUM score of its list: the
// k-th largest of those maxima bounds the final k-th best from below, which lets
// topk_merge.cu fold the 2368 lists in ONE launch (merge_select_kernel).
//
// Algorithmic HBM traffic: ntotal * dpad * 2 bytes per pass (SURVEY.md 8d).
#include "index.cuh"

namespace ivr {

constexpr int kStreamThreads = 256;            // 8 warps
constexpr int kStreamWarps   = kStreamThreads / 32;
constexpr int kStreamCtasPerSm = 2;
constexpr int kStreamMaxNq   = 4;
constexpr int kRowsPerStep   = 4;              // 8 lanes per row
constexpr int kUnroll        = 2;              // steps in flight

template <int NQ, int DCH, int E>
__global__ void __launch_bounds__(kStreamThreads, kStreamCtasPerSm)
search_stream_kernel(const __half* __restrict__ rows, int64_t n_rows, int dpad,
                     const float* __restrict__ q,      // [nq_real, dim] fp32, as the caller passed them
                     int dim, int nq_real,
                     int k, int C, uint64_t* __restrict__ lists, int* __restrict__ counts,
                     uint32_t* __restrict__ maxima) {
    extern __shared__ float s_q[];                     // NQ * dpad
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane & 7, rgrp = lane >> 3;
    const int nch = (DCH > 0) ? DCH : dpad / 64;       // 64-element chunks per row

    // queries -> shared memory, zero-padded to dpad columns / NQ rows (no separate padding launch)
    for (int i = threadIdx.x; i < NQ * dpad; i += blockDim.x) {
        const int r = i / dpad, c = i - r * dpad;
        s_q[i] = (r < nq_real && c < dim) ? q[static_cast<int64_t>(r) * dim + c] : 0.f;
    }
    __syncthreads();

    const int64_t gw = static_cast<int64_t>(blockIdx.x) * kStreamWarps + warp;
    const int64_t nw = static_cast<int64_t>(gridDim.x) * kStreamWarps;
    // groups of kUnroll steps (8 rows) dealt round-robin to the warps of the grid
    const int64_t steps_total = (n_rows + kRowsPerStep - 1) / kRowsPerStep;
    const int64_t s1 = steps_total;

    uint64_t* my_lists = lists + gw * NQ * C;
    int   cnt[NQ];
    float tau[NQ];
#pragma unroll
    for (int i = 0; i < NQ; ++i) { cnt[i] = 0; tau[i] = __int_as_float(0xff800000); }

    for (int64_t s = gw * kUnroll; s < s1; s += nw * kUnroll) {
        float acc[kUnroll][NQ];
        int64_t row[kUnroll];
        uint4 x[kUnroll][(DCH > 0) ? DCH : 1];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            row[u] = (s + u) * kRowsPerStep + rgrp;
            const bool ok = (s + u) < s1 && row[u] < n_rows;
            if (!ok) row[u] = -1;
#pragma unroll
            for (int i = 0; i < NQ; ++i) acc[u][i] = 0.f;
        }
        if (DCH > 0) {
            // issue every load of both steps before the first use
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const __half* rp = rows + (row[u] < 0 ? 0 : row[u]) * dpad + sub * 8;
#pragma unroll
                for (int c = 0; c < ((DCH > 0) ? DCH : 1); ++c)
                    x[u][c] = (row[u] >= 0) ? ldg_nc_v4(rp + c * 64) : make_uint4(0, 0, 0, 0);
            }
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
#pragma unroll
                for (int c = 0; c < ((DCH > 0) ? DCH : 1); ++c) {
                    const uint4 v = x[u][c];
                    const float2 p0 = h2f2(v.x), p1 = h2f2(v.y), p2 = h2f2(v.z), p3 = h2f2(v.w);
                    const float f0 = p0.x, f1 = p0.y, f2 = p1.x, f3 = p1.y, f4 = p2.x, f5 = p2.y, f6 = p3.x, f7 = p3.y;
#pragma unroll
                    for (int i = 0; i < NQ; ++i) {
                        const float4 qa = *reinterpret_cast<const float4*>(s_q + i * dpad + c * 64 + sub * 8);
                        const float4 qb = *reinterpret_cast<const float4*>(s_q + i * dpad + c * 64 + sub * 8 + 4);
                        float a = acc[u][i];
                        a = fmaf(f0, qa.x, a); a = fmaf(f1, qa.y, a); a = fmaf(f2, qa.z, a); a = fmaf(f3, qa.w, a);
                        a = fmaf(f4, qb.x, a); a = fmaf(f5, qb.y, a); a = fmaf(f6, qb.z, a); a = fmaf(f7, qb.w, a);
                        acc[u][i] = a;
                    }
                }
            }
        } else {
            for (int c = 0; c < nch; ++c) {
#pragma unroll
                for (int u = 0; u < kUnroll; ++u) {
                    const __half* rp = rows + (row[u] < 0 ? 0 : row[u]) * dpad + sub * 8;
                    const uint4 v = (row[u] >= 0) ? ldg_nc_v4(rp + c * 64) : make_uint4(0, 0, 0, 0);
                    const float2 p0 = h2f2(v.x), p1 = h2f2(v.y), p2 = h2f2(v.z), p3 = h2f2(v.w);
                    const float f0 = p0.x, f1 = p0.y, f2 = p1.x, f3 = p1.y, f4 = p2.x, f5 = p2.y, f6 = p3.x, f7 = p3.y;
#pragma unroll
                    for (int i = 0; i < NQ; ++i) {
                        const float4 qa = *reinterpret_cast<const float4*>(s_q + i * dpad + c * 64 + sub * 8);
                        const float4 qb = *reinterpret_cast<const float4*>(s_q + i * dpad + c * 64 + sub * 8 + 4);
                        float a = acc[u][i];
                        a = fmaf(f0, qa.x, a); a = fmaf(f1, qa.y, a); a = fmaf(f2, qa.z, a); a = fmaf(f3, qa.w, a);
                        a = fmaf(f4, qb.x, a); a = fmaf(f5, qb.y, a); a = fmaf(f6, qb.z, a); a = fmaf(f7, qb.w, a);
                        acc[u][i] = a;
                    }
                }
            }
        }
        // reduce over the 8 lanes of each row
#pragma unroll
        for (int u = 0; u < kUnroll; ++u)
#pragma unroll
            for (int i = 0; i < NQ; ++i) {
                float a = acc[u][i];
                a += __shfl_xor_sync(0xffffffffu, a, 1);
                a += __shfl_xor_sync(0xffffffffu, a, 2);
                a += __shfl_xor_sync(0xffffffffu, a, 4);
                acc[u][i] = a;
            }
        // admit candidates (lane sub==0 of each row speaks for the row)
#pragma unroll
        for (int i = 0; i < NQ; ++i) {
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const bool pass = (sub == 0) && (row[u] >= 0) && (acc[u][i] > tau[i]);
                const unsigned m = __ballot_sync(0xffffffffu, pass);
                if (pass) {
                    const int pos = cnt[i] + __popc(m & ((1u << lane) - 1u));
                    my_lists[i * C + pos] = make_key(acc[u][i], static_cast<uint32_t>(row[u]));
                }
                cnt[i] += __popc(m);
            }
            if (cnt[i] > C - kRowsPerStep * kUnroll) {          // warp-uniform
                __syncwarp();
                tau[i] = warp_compact<E>(my_lists + i * C, cnt[i], k, C, lane);
                cnt[i] = min(cnt[i], k);
            }
        }
    }
    // the list is left as it is (up to C entries: the merge filters it); publish its size and its maximum score
    __syncwarp();
#pragma unroll
    for (int i = 0; i < NQ; ++i) {
        uint32_t mx = 0;
        for (int j = lane; j < cnt[i]; j += 32) mx = max(mx, static_cast<uint32_t>(my_lists[i * C + j] >> 32));
        mx = __reduce_max_sync(0xffffffffu, mx);
        if (lane == 0) { counts[gw * NQ + i] = cnt[i]; maxima[gw * NQ + i] = mx; }
    }
}

template <int NQ, int E>
static int launch_stream(ivr_index* idx, const float* q, int nq_real, int k, int C, uint64_t* lists, int* counts,
                         uint32_t* maxima, int grid, cudaStream_t st) {
    const size_t smem = static_cast<size_t>(NQ) * idx->dpad * sizeof(float);
    const int dch = idx->dpad / 64;
#define IVR_LAUNCH_STREAM(DCH)                                                                     \
    do {                                                                                           \
        auto kern = search_stream_kernel<NQ, DCH, E>;                                              \
        if (smem > 48 * 1024)                                                                      \
            IVR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,       \
                                          static_cast<int>(smem)));                                \
        kern<<<grid, kStreamThreads, smem, st>>>(idx->rows, idx->ntotal, idx->dpad, q, idx->dim,   \
                                                 nq_real, k, C, lists, counts, maxima);            \
    } while (0)
    switch (dch) {
        case 8:  IVR_LAUNCH_STREAM(8);  break;     // 512  (CLIP ViT-B/32)
        case 12: IVR_LAUNCH_STREAM(12); break;     // 768  (CLIP ViT-L/14)
        default: IVR_LAUNCH_STREAM(0);  break;     // any other multiple of 64
    }
#undef IVR_LAUNCH_STREAM
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

template <int E>
static int launch_stream_nq(ivr_index* idx, int nq, int nq_real, const float* q, int k, int C, uint64_t* lists,
                            int* counts, uint32_t* maxima, int grid, cudaStream_t st) {
    switch (nq) {                                  // nq == 3 runs as 4 with a zero query
        case 1: return launch_stream<1, E>(idx, q, nq_real, k, C, lists, counts, maxima, grid, st);
        case 2: return launch_stream<2, E>(idx, q, nq_real, k, C, lists, counts, maxima, grid, st);
        default: return launch_stream<4, E>(idx, q, nq_real, k, C, lists, counts, maxima, grid, st);
    }
}

int search_stream(ivr_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev,
                  int64_t* I_dev, int64_t id_offset, cudaStream_t st) {
    const int kcap = kcap_for(k);
    const int C = 2 * kcap;
    const int grid = idx->sm_count * kStreamCtasPerSm;
    const int64_t n_lists = static_cast<int64_t>(grid) * kStreamWarps;

    // workspace carve-up
    const size_t list_keys = static_cast<size_t>(n_lists) * kStreamMaxNq * C;
    const size_t tmp_keys = merge_tmp_entries(static_cast<int>(n_lists), kStreamMaxNq, k);
    const size_t cnt_ints = static_cast<size_t>(n_lists) * kStreamMaxNq * 2 + 1024;
    const bool select = k <= kSelectMaxK;             // one-launch merge by the list-maxima bound; exact radix levels above
    Carve carve;
    const size_t o_l = carve(list_keys * 8), o_t = carve(tmp_keys * 8),
                 o_c = carve(cnt_ints * 4), o_m = carve(static_cast<size_t>(n_lists) * kStreamMaxNq * 4),
                 o_p = carve(static_cast<size_t>(kStreamMaxNq) * kSelectPoolCap * 8);
    IVR_TRY(ensure_ws(idx, carve.size));
    char* ws = static_cast<char*>(idx->ws);
    uint64_t* lists = reinterpret_cast<uint64_t*>(ws + o_l);
    uint64_t* tmp = reinterpret_cast<uint64_t*>(ws + o_t);
    int* counts = reinterpret_cast<int*>(ws + o_c);
    int* tmp_counts = counts + n_lists * kStreamMaxNq;
    uint32_t* maxima = reinterpret_cast<uint32_t*>(ws + o_m);
    uint64_t* pool = reinterpret_cast<uint64_t*>(ws + o_p);
    int* merge_state = idx->sel_state;                        // [kStreamMaxNq] pool counters, [kStreamMaxNq] tickets: zero between calls

    for (int64_t q0 = 0; q0 < nq; q0 += kStreamMaxNq) {
        const int b_real = static_cast<int>(nq - q0 < kStreamMaxNq ? nq - q0 : kStreamMaxNq);
        const int b = (b_real == 3) ? 4 : b_real;             // kernel batch (3 is padded to 4)
        const bool timed = idx->timing && q0 == 0;         // the first batch; the kernel reads fp32 queries: no prep
        timing_mark(idx, timed, kPrepBegin, st); timing_mark(idx, timed, kPrepEnd, st); timing_mark(idx, timed, kScoreBegin, st);
        int rc;
        switch (kcap) {
            case 128: rc = launch_stream_nq<8>(idx, b, b_real, q_dev + q0 * idx->dim, k, C, lists, counts, maxima, grid, st); break;   // k <= 128: register sort
            default:  rc = launch_stream_nq<0>(idx, b, b_real, q_dev + q0 * idx->dim, k, C, lists, counts, maxima, grid, st); break;   // larger k: in-memory sort
        }
        IVR_TRY(rc);
        idx->launches[0]++;
        timing_mark(idx, timed, kScoreEnd, st); timing_mark(idx, timed, kMergeBegin, st);
        MergeIn in{};
        in.entries = lists; in.counts = counts;
        in.list_stride = static_cast<int64_t>(b) * C; in.q_stride = C;
        in.cnt_list_stride = b; in.cnt_q_stride = 1;
        in.n_lists = static_cast<int>(n_lists); in.fixed_count = 0;
        if (select)
            IVR_TRY(merge_select_final(in, maxima, b_real, k, D_dev ? D_dev + q0 * k : nullptr, I_dev + q0 * k, id_offset,
                                       pool, merge_state, merge_state + kStreamMaxNq, idx->sm_count, st, &idx->launches[1]));
        else
            IVR_TRY(merge_lists_final(in, b_real, k, D_dev ? D_dev + q0 * k : nullptr, I_dev + q0 * k, id_offset, tmp,
                                      tmp_counts, st, &idx->launches[1]));
        timing_mark(idx, timed, kMergeEnd, st);
    }
    if (idx->timing) idx->ev_valid[0] = idx->ev_valid[1] = idx->ev_valid[2] = true;
    return IVR_OK;
}

}  // namespace ivr

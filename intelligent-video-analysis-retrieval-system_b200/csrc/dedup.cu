// dedup.cu -- K4: fused normalise-and-compare kernels for near-duplicate pruning.
//
// Reference rules replaced (all cosines are sklearn.metrics.pairwise.cosine_similarity
// on two 1xD float32 rows: normalise each row, then dot):
//   filter.calculate_similarities            filter.py:142-151   (consecutive cosine)
//   filter.filter_similar_frames_advanced    filter.py:224-259   (window rule)
//   filter.filter_similar_frames_in_scene    filter.py:178-222   (last-kept chain)
//   video_frame_filter rule                  video_frame_filter.py:63-70
//
// banded_cosine_kernel: ONE pass over the fp32 frame matrix (HBM-bound, D*4 bytes
// per frame).  Each warp owns one frame per batch: it loads the row with 128-bit
// coalesced loads, normalises it in registers, parks the normalised row in a
// shared-memory ring, and dots it against the previous W parked rows.  Output per
// frame: a W-bit mask (bit d-1 <=> cos(e_i, e_{i-d}) >= thr) and cos(e_i, e_{i-1}).
// window_resolve_kernel then runs the reference's sequential greedy rule per scene
// on the bit masks alone (O(1) per frame with a W-bit keep history).
#include "common.cuh"

#include <cstdlib>

namespace ivr {

constexpr int kDedupWarps = 8;                 // frames per batch and per CTA
constexpr int kDedupThreads = kDedupWarps * 32;

// DV > 0: d == DV*128, each lane holds DV float4 of its row.  DV == 0: generic d.
template <int DV>
__global__ void __launch_bounds__(kDedupThreads)
banded_cosine_kernel(const float* __restrict__ e, int64_t n, int64_t out_begin, int d, int window, float thr,
                     uint32_t* __restrict__ masks, float* __restrict__ cos_prev, int ring) {
    extern __shared__ float s_ring[];          // ring * dstride floats
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int dstride = (DV > 0) ? DV * 128 : ((d + 3) / 4 * 4);

    // contiguous chunk of the output frames [out_begin, n) per CTA (+ a halo of `window` frames re-normalised
    // locally; frames before out_begin are context only -- the chunked host path re-uses the tail of the last chunk)
    const int64_t span = n - out_begin;
    const int64_t f0 = out_begin + span * blockIdx.x / gridDim.x, f1 = out_begin + span * (blockIdx.x + 1) / gridDim.x;
    if (f0 >= f1) return;
    const int64_t fs = (f0 - window > 0) ? f0 - window : 0;

    constexpr int NV = (DV > 0) ? DV : 1;
    float4 cur[NV], nxt[NV];

    auto load_row = [&](int64_t i, float4 (&r)[NV]) {
        if (DV > 0) {
            const float4* p = reinterpret_cast<const float4*>(e + i * d);
#pragma unroll
            for (int j = 0; j < NV; ++j) r[j] = ldg_nc_f4(p + lane + 32 * j);
        }
    };

    int64_t base = fs;
    if (DV > 0 && base + warp < f1) load_row(base + warp, nxt);

    for (; base < f1; base += kDedupWarps) {
        const int64_t i = base + warp;
        const bool live = i < f1;
        float* slot = s_ring + static_cast<size_t>((i % ring)) * dstride;
        if (live) {
            if (DV > 0) {
#pragma unroll
                for (int j = 0; j < NV; ++j) cur[j] = nxt[j];
                if (i + kDedupWarps < f1) load_row(i + kDedupWarps, nxt);   // prefetch next batch
                float ss = 0.f;
#pragma unroll
                for (int j = 0; j < NV; ++j) {
                    ss = fmaf(cur[j].x, cur[j].x, ss); ss = fmaf(cur[j].y, cur[j].y, ss);
                    ss = fmaf(cur[j].z, cur[j].z, ss); ss = fmaf(cur[j].w, cur[j].w, ss);
                }
                for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
                float nrm = sqrtf(ss);
                if (nrm == 0.f) nrm = 1.f;                                   // sklearn: 0 -> 1
                const float inv = 1.0f / nrm;
#pragma unroll
                for (int j = 0; j < NV; ++j) {
                    cur[j].x *= inv; cur[j].y *= inv; cur[j].z *= inv; cur[j].w *= inv;
                    reinterpret_cast<float4*>(slot)[lane + 32 * j] = cur[j];
                }
            } else {
                const float* p = e + i * d;
                float ss = 0.f;
                for (int c = lane; c < d; c += 32) { const float v = p[c]; ss = fmaf(v, v, ss); }
                for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
                float nrm = sqrtf(ss);
                if (nrm == 0.f) nrm = 1.f;
                for (int c = lane; c < d; c += 32) slot[c] = p[c] / nrm;
            }
        }
        __syncthreads();
        if (live && i >= f0) {
            uint32_t m = 0;
            float c1 = 1.0f;
            for (int dd = 1; dd <= window; ++dd) {
                const int64_t j = i - dd;
                if (j < 0) break;
                const float* other = s_ring + static_cast<size_t>((j % ring)) * dstride;
                float acc = 0.f;
                if (DV > 0) {
#pragma unroll
                    for (int jj = 0; jj < NV; ++jj) {
                        const float4 o = reinterpret_cast<const float4*>(other)[lane + 32 * jj];
                        acc = fmaf(cur[jj].x, o.x, acc); acc = fmaf(cur[jj].y, o.y, acc);
                        acc = fmaf(cur[jj].z, o.z, acc); acc = fmaf(cur[jj].w, o.w, acc);
                    }
                } else {
                    for (int c = lane; c < d; c += 32) acc = fmaf(slot[c], other[c], acc);
                }
                for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                if (acc >= thr) m |= 1u << (dd - 1);
                if (dd == 1) c1 = acc;
            }
            if (lane == 0) {
                if (masks) masks[i] = m;
                if (cos_prev) cos_prev[i] = c1;
            }
        }
        // ring holds window + 2 batches: the next batch's writes cannot touch rows this
        // batch still reads, so one barrier per batch is enough.
    }
}

// ---------------------------------------------------------------------------
// Register-window variant (window <= 8, d in {384, 512}) -- the default for those shapes.
// Every WARP walks its own contiguous run of frames sequentially and keeps the last 8 normalised
// rows in REGISTERS (the frame loop is unrolled by 8, so the window slot of a frame is a
// compile-time index).  Frames are prefetched 7 deep with cp.async into a private per-warp staging
// ring (each lane copies and later reads only its own 16-byte chunks, so no warp or CTA barrier is
// ever needed).  Per frame: 4-6 LDS.128, 128 x DV/4... FMAs against the register window, one
// 9-shuffle transpose-reduction of the 8 dot products, one ballot.  No shared-memory ring of
// normalised rows, no __syncthreads: the kernel is a pure HBM stream.
// ---------------------------------------------------------------------------
constexpr int kRwWarps = 4;
constexpr int kRwSlots = 8;                     // staged frames per warp
constexpr int kRwWindow = 8;

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                 ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst))), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Packed fp32 pairs (sm_100 FFMA2 / FMUL2): two IEEE fp32 operations per issued instruction.  The register-window
// kernel is bound by instruction issue (ncu: 69 % issue-active, 144 of ~230 instructions per frame are FMAs), not
// by the FP32 pipe or HBM, so halving the FMA instruction count is what moves it.
__device__ __forceinline__ void ffma2(float& c0, float& c1, float a0, float a1, float b0, float b1) {
    asm("{\n\t.reg .b64 ra, rb, rc;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%0, %1};\n\t"
        "fma.rn.f32x2 rc, ra, rb, rc;\n\tmov.b64 {%0, %1}, rc;\n\t}"
        : "+f"(c0), "+f"(c1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}
__device__ __forceinline__ void fmul2(float& c0, float& c1, float a0, float a1, float b0, float b1) {
    asm("{\n\t.reg .b64 ra, rb, rc;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "mul.rn.f32x2 rc, ra, rb;\n\tmov.b64 {%0, %1}, rc;\n\t}"
        : "=f"(c0), "=f"(c1) : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}

template <int DV>
__global__ void __launch_bounds__(kRwWarps * 32, 3)
banded_cosine_rw_kernel(const float* __restrict__ e, int64_t n, int64_t out_begin, int window, float thr,
                        uint32_t* __restrict__ masks, float* __restrict__ cos_prev) {
    extern __shared__ float4 s_stage[];         // [kRwWarps][kRwSlots][DV * 32]
    constexpr int RS4 = DV * 32;                // float4 per row
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t gw = static_cast<int64_t>(blockIdx.x) * kRwWarps + warp;
    const int64_t nw = static_cast<int64_t>(gridDim.x) * kRwWarps;
    const int64_t span = n - out_begin;         // frames before out_begin are context only (chunked host path)
    const int64_t f0 = out_begin + span * gw / nw, f1 = out_begin + span * (gw + 1) / nw;
    if (f0 >= f1) return;                        // no CTA-wide barrier anywhere below
    const int64_t fs = (f0 - kRwWindow > 0) ? f0 - kRwWindow : 0;
    // everything inside the frame loop is 32-bit and relative to fs (the kernel is bound by instruction issue)
    const int total = static_cast<int>(f1 - fs);                     // frames this warp walks, halo included
    const int first_out = static_cast<int>(f0 - fs);                 // first local frame that produces output
    const int before = static_cast<int>(fs < kRwWindow ? fs : kRwWindow);   // real predecessors of local frame 0, capped
    float4* const stage = s_stage + static_cast<size_t>(warp) * kRwSlots * RS4 + lane;   // this lane's column of the ring
    const float4* pf = reinterpret_cast<const float4*>(e) + fs * RS4 + lane;             // next frame to prefetch
    uint32_t* const mout = masks ? masks + fs : nullptr;
    float* const cout = cos_prev ? cos_prev + fs : nullptr;
    const int dd = (lane & 7) + 1;                                   // the look-back this lane reports (lanes 0..7 count)

    auto issue = [&](int t, int slot) {
        if (t < total) {
#pragma unroll
            for (int j = 0; j < DV; ++j) cp_async16(stage + slot * RS4 + 32 * j, pf + 32 * j);
        }
        pf += RS4;
        cp_async_commit();                      // always commit: keeps the group count uniform
    };
#pragma unroll
    for (int x = 0; x < kRwSlots - 1; ++x) issue(x, x);

    float4 win[kRwWindow][DV];
#pragma unroll
    for (int w = 0; w < kRwWindow; ++w)
#pragma unroll
        for (int j = 0; j < DV; ++j) win[w][j] = make_float4(0.f, 0.f, 0.f, 0.f);

    for (int t0 = 0; t0 < total; t0 += kRwWindow) {
#pragma unroll
        for (int u = 0; u < kRwWindow; ++u) {
            const int t = t0 + u;
            if (t < total) {                                                // warp-uniform
                cp_async_wait<kRwSlots - 2>();                              // frame t has landed
                float4 cur[DV];
#pragma unroll
                for (int j = 0; j < DV; ++j) cur[j] = stage[u * RS4 + 32 * j];
                issue(t + kRwSlots - 1, (u + kRwSlots - 1) % kRwSlots);    // refill the slot read one step ago
                // The 8 dot products are taken with the RAW row and scaled by 1/||row|| afterwards
                // (dot(x/|x|, w) == dot(x, w)/|x| up to one rounding), so the norm reduction and the
                // dot reduction are two independent shuffle chains instead of one long one.
                float ss0 = 0.f, ss1 = 0.f;                                 // even / odd partial sums (FFMA2)
#pragma unroll
                for (int j = 0; j < DV; ++j) {
                    ffma2(ss0, ss1, cur[j].x, cur[j].y, cur[j].x, cur[j].y);
                    ffma2(ss0, ss1, cur[j].z, cur[j].w, cur[j].z, cur[j].w);
                }
                float ss = ss0 + ss1;
                float acc[kRwWindow];
#pragma unroll
                for (int d1 = 1; d1 <= kRwWindow; ++d1) {
                    const int w = (u - d1 + 2 * kRwWindow) % kRwWindow;     // slot of frame t - d1
                    float a0 = 0.f, a1 = 0.f;
#pragma unroll
                    for (int j = 0; j < DV; ++j) {
                        ffma2(a0, a1, cur[j].x, cur[j].y, win[w][j].x, win[w][j].y);
                        ffma2(a0, a1, cur[j].z, cur[j].w, win[w][j].z, win[w][j].w);
                    }
                    acc[d1 - 1] = a0 + a1;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
                // transpose-reduce the 8 sums: lane bit 2 picks index bit 2, bit 1 -> bit 1, bit 0 -> bit 0, so lane l
                // ends with the partial of index l & 7; two more exchanges add the four 8-lane groups together
#pragma unroll
                for (int s2 = 4, half = 4; half > 0; s2 >>= 1, half >>= 1) {
                    const bool up = (lane & s2) != 0;
#pragma unroll
                    for (int a = 0; a < half; ++a) {
                        const float send = up ? acc[a] : acc[a + half];
                        const float keep = up ? acc[a + half] : acc[a];
                        acc[a] = keep + __shfl_xor_sync(0xffffffffu, send, s2);
                    }
                }
                float val = acc[0];
                val += __shfl_xor_sync(0xffffffffu, val, 8);
                val += __shfl_xor_sync(0xffffffffu, val, 16);
                // 1 / ||row||: reciprocal square root + one Newton step while ss is a normal fp32 below 2^126 (there
                // inv * inv neither overflows nor goes subnormal).  Outside that range -- zero, subnormal, overflowed
                // to inf, NaN -- take sklearn's 1 / sqrt(ss) with a zero norm mapped to 1: an overflowed norm gives
                // cosine 0, not NaN.  ss is the same on every lane after the xor butterfly: the branch is warp-uniform.
                // (The dots above use the raw row: a row whose norm itself exceeds FLT_MAX still overflows them.)
                float inv;
                if (ss >= 0x1p-126f && ss < 0x1p126f) {
                    inv = rsqrtf(ss);
                    inv = inv * fmaf(-0.5f * ss, inv * inv, 1.5f);
                } else {
                    inv = (ss == 0.f) ? 1.f : 1.0f / sqrtf(ss);
                }
                val *= inv;
#pragma unroll
                for (int j = 0; j < DV; ++j) {                              // frame t (normalised) replaces frame t - 8
                    fmul2(win[u][j].x, win[u][j].y, cur[j].x, cur[j].y, inv, inv);
                    fmul2(win[u][j].z, win[u][j].w, cur[j].z, cur[j].w, inv, inv);
                }
                const bool ge = dd <= min(window, before + t) && val >= thr;   // only real predecessors inside the window
                const unsigned ballot = __ballot_sync(0xffffffffu, ge);
                if (t >= first_out && lane == 0) {
                    if (mout) mout[t] = ballot & 0xffu;                     // lanes 0..7 hold look-backs 1..8
                    if (cout) cout[t] = (before + t >= 1) ? val : 1.0f;
                }
            }
        }
    }
    cp_async_wait<0>();
}

// One thread per scene: the reference's greedy rule on the bit masks.
//   keep_i = !exists d in [1, min(window, i - scene_start)] : keep_{i-d} && bit_{d-1}(mask_i)
__global__ void window_resolve_kernel(const uint32_t* __restrict__ masks,
                                      const int64_t* __restrict__ scene_start,
                                      const int64_t* __restrict__ scene_end, int64_t n_scenes,
                                      int64_t n, int window, uint8_t* __restrict__ keep) {
    const int64_t s = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (s >= n_scenes) return;
    int64_t a = scene_start[s], b = scene_end[s];
    if (a < 0) a = 0;
    if (b >= n) b = n - 1;
    const uint32_t wmask = (window >= 32) ? 0xffffffffu : ((1u << window) - 1u);
    uint32_t hist = 0;                          // bit d-1 = keep flag of frame i-d (this scene only)
    for (int64_t i = a; i <= b; ++i) {
        const uint32_t k = ((masks[i] & hist & wmask) == 0u) ? 1u : 0u;
        keep[i] = static_cast<uint8_t>(k);
        hist = (hist << 1) | k;                 // frames before the scene start are never set
    }
}

// Scene split AND greedy rule in one pass over the per-frame outputs of the banded kernel -- the device form of
// detect_scene_transitions + group_into_scenes + filter_similar_frames_advanced per scene (filter.py:153-176, 224-315):
// frame i starts a scene iff i == 0 or cos(e_i, e_{i-1}) < transition_thr (strict); a scene runs to the frame before
// the next start; scenes shorter than min_len vanish (keep = 0); inside a scene the window rule runs on the masks.
// One thread per frame; only scene-start threads do work (they walk their own scene: mean length ~20 frames).
__global__ void scene_resolve_kernel(const uint32_t* __restrict__ masks, const float* __restrict__ cos_prev, int64_t n,
                                     int window, float transition_thr, int min_len, uint8_t* __restrict__ keep,
                                     unsigned long long* __restrict__ stats) {   // [scenes kept, frames inside them]
    const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (i >= n) return;
    if (i != 0 && !(cos_prev[i] < transition_thr)) return;          // not a scene start
    int64_t end = i + 1;
    while (end < n && !(cos_prev[end] < transition_thr)) ++end;     // [i, end) is the scene
    if (end - i < min_len) {
        for (int64_t j = i; j < end; ++j) keep[j] = 0;
        return;
    }
    if (stats) { atomicAdd(stats, 1ull); atomicAdd(stats + 1, static_cast<unsigned long long>(end - i)); }
    const uint32_t wmask = (window >= 32) ? 0xffffffffu : ((1u << window) - 1u);
    uint32_t hist = 0;                          // bit d-1 = keep flag of frame j-d (this scene only)
    for (int64_t j = i; j < end; ++j) {
        const uint32_t kf = (window <= 0 || (masks[j] & hist & wmask) == 0u) ? 1u : 0u;   // empty window keeps everything
        keep[j] = static_cast<uint8_t>(kf);
        hist = (hist << 1) | kf;
    }
}

int launch_scene_resolve(const uint32_t* masks, const float* cos_prev, int64_t n, int window, float transition_thr,
                         int min_len, uint8_t* keep, unsigned long long* stats, cudaStream_t st) {
    if (n <= 0) return IVR_OK;
    const int threads = 256;
    scene_resolve_kernel<<<static_cast<unsigned>((n + threads - 1) / threads), threads, 0, st>>>(
        masks, cos_prev, n, window, transition_thr, min_len, keep, stats);
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

// One warp per scene: keep-chain rules with unbounded look-back in frame index.
//   fifo == 1 : last-kept chain (filter.py:178-222; video_frame_filter.py:63-70): keep i iff
//               i - last_kept >= min_distance and cos(e_i, e_last_kept) < thr; with force_last the
//               scene's last frame is always kept.
//   fifo  > 1 : FIFO of the last `fifo` KEPT frames (filter_research_update.py:316-338, Phase 4):
//               keep i iff cos(e_i, e_p) < thr for every p in the FIFO.
constexpr int kMaxFifo = 16;

__global__ void chain_resolve_kernel(const float* __restrict__ e, int d,
                                     const int64_t* __restrict__ scene_start,
                                     const int64_t* __restrict__ scene_end, int64_t n_scenes,
                                     int64_t n, int min_distance, float thr, int force_last, int fifo,
                                     uint8_t* __restrict__ keep) {
    const int lane = threadIdx.x & 31;
    const int64_t s = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
    if (s >= n_scenes) return;
    int64_t a = scene_start[s], b = scene_end[s];
    if (a < 0) a = 0;
    if (b >= n) b = n - 1;
    if (a > b) return;
    auto norm_of = [&](int64_t i) {
        const float* p = e + i * d;
        float ss = 0.f;
        for (int c = lane; c < d; c += 32) { const float v = p[c]; ss = fmaf(v, v, ss); }
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        float nrm = sqrtf(ss);
        return nrm == 0.f ? 1.f : nrm;
    };
    // FIFO of kept frames: index + norm, oldest first (warp-uniform registers)
    int64_t kept_idx[kMaxFifo];
    float kept_nrm[kMaxFifo];
    int nk = 1;
    kept_idx[0] = a; kept_nrm[0] = norm_of(a);
    int64_t last = a;
    if (lane == 0) keep[a] = 1;
    for (int64_t i = a + 1; i <= b; ++i) {
        if (i - last < min_distance) { if (lane == 0) keep[i] = 0; continue; }
        const float ni = norm_of(i);
        const float* p = e + i * d;
        bool unique = true;
        for (int w = 0; w < nk && unique; ++w) {                 // oldest first, stop at the first hit
            const float* q = e + kept_idx[w] * d;
            const float nq = kept_nrm[w];
            float acc = 0.f;
            for (int c = lane; c < d; c += 32) acc = fmaf(p[c] / ni, q[c] / nq, acc);
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (!(acc < thr)) unique = false;
        }
        if (lane == 0) keep[i] = unique ? 1 : 0;
        if (unique) {
            last = i;
            if (nk == fifo) {                                     // pop the oldest
#pragma unroll
                for (int w = 0; w + 1 < kMaxFifo; ++w) { kept_idx[w] = kept_idx[w + 1]; kept_nrm[w] = kept_nrm[w + 1]; }
                --nk;
            }
            kept_idx[nk] = i; kept_nrm[nk] = ni; ++nk;
        }
    }
    if (force_last && last != b && lane == 0) keep[b] = 1;
}

// ---------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------
static thread_local bool        g_dedup_timing = false;
static thread_local cudaEvent_t g_dedup_ev[4] = {nullptr, nullptr, nullptr, nullptr};
static thread_local bool        g_dedup_ev_valid = false;

int dedup_set_timing(int enable) { g_dedup_timing = enable != 0; return IVR_OK; }

int dedup_last_timing(float ms[2]) {
    if (!g_dedup_ev_valid) { set_error("no timed dedup call on this thread"); return IVR_EINVAL; }
    IVR_CUDA(cudaEventSynchronize(g_dedup_ev[3]));
    IVR_CUDA(cudaEventElapsedTime(&ms[0], g_dedup_ev[0], g_dedup_ev[1]));
    IVR_CUDA(cudaEventElapsedTime(&ms[1], g_dedup_ev[2], g_dedup_ev[3]));
    return IVR_OK;
}

static int env_flag(const char* name, int dflt) {
    const char* e = getenv(name);
    return (e && *e) ? atoi(e) : dflt;
}

int launch_banded(const float* e_dev, int64_t n, int64_t out_begin, int d, int window, float thr, uint32_t* masks,
                  float* cos_prev, int sm_count, cudaStream_t st) {
    // Masks / cosines are produced for frames [out_begin, n); frames before out_begin are look-back context only.
    if (n <= out_begin) return IVR_OK;
    const int64_t span = n - out_begin;
    const bool aligned = (reinterpret_cast<uintptr_t>(e_dev) & 15) == 0;
    // IVR_DEDUP_KERNEL: 0 = register-window kernel (default for window <= 8, d = 384/512), 2 = generic kernel
    const int variant = env_flag("IVR_DEDUP_KERNEL", 0);
    if (aligned && window <= kRwWindow && (d == 512 || d == 384) && variant == 0) {
        const size_t smem = static_cast<size_t>(kRwWarps) * kRwSlots * d * sizeof(float);
        int64_t grid = static_cast<int64_t>(sm_count) * 3;                  // persistent: 3 CTAs per SM
        const int64_t max_grid = (span + 255) / 256;
        if (grid > max_grid) grid = max_grid;
        if (grid < 1) grid = 1;
        if (d == 512) {
            auto kern = banded_cosine_rw_kernel<4>;
            IVR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
            kern<<<static_cast<unsigned>(grid), kRwWarps * 32, smem, st>>>(e_dev, n, out_begin, window, thr, masks, cos_prev);
        } else {
            auto kern = banded_cosine_rw_kernel<3>;
            IVR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
            kern<<<static_cast<unsigned>(grid), kRwWarps * 32, smem, st>>>(e_dev, n, out_begin, window, thr, masks, cos_prev);
        }
        IVR_CUDA(cudaGetLastError());
        return IVR_OK;
    }
    const int ring = window + 2 * kDedupWarps;
    int dv = 0;
    if (d % 128 == 0 && aligned) dv = d / 128;
    const int dstride = dv ? d : (d + 3) / 4 * 4;
    const size_t smem = static_cast<size_t>(ring) * dstride * sizeof(float);
    if (smem > 227 * 1024) {
        set_error("dedup: window %d x dim %d needs %zu B of shared memory (> 227 KB)", window, d, smem);
        return IVR_EUNSUPPORTED;
    }
    // enough CTAs to fill the machine twice over, but chunks of at least 64 frames so the
    // re-normalised halo stays a small fraction of the work
    int64_t grid = static_cast<int64_t>(sm_count) * 4;
    const int64_t max_grid = (span + 63) / 64;
    if (grid > max_grid) grid = max_grid;
    if (grid < 1) grid = 1;
#define IVR_LAUNCH_BANDED(DV)                                                                      \
    do {                                                                                           \
        auto kern = banded_cosine_kernel<DV>;                                                      \
        if (smem > 48 * 1024)                                                                      \
            IVR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,       \
                                          static_cast<int>(smem)));                                \
        kern<<<static_cast<unsigned>(grid), kDedupThreads, smem, st>>>(e_dev, n, out_begin, d, window, thr,  \
                                                                       masks, cos_prev, ring);     \
    } while (0)
    switch (dv) {
        case 3: IVR_LAUNCH_BANDED(3); break;     // 384
        case 4: IVR_LAUNCH_BANDED(4); break;     // 512
        case 6: IVR_LAUNCH_BANDED(6); break;     // 768
        case 8: IVR_LAUNCH_BANDED(8); break;     // 1024
        default: IVR_LAUNCH_BANDED(0); break;
    }
#undef IVR_LAUNCH_BANDED
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

int dedup_window_device(int device, const float* e_dev, int64_t n, int d,
                        const int64_t* scene_start_dev, const int64_t* scene_end_dev,
                        int64_t n_scenes, int window, float thr, uint8_t* keep_dev,
                        float* cos_prev_dev, uint32_t* mask_ws_dev, cudaStream_t st) {
    if (n <= 0) return IVR_OK;
    int sm_count = 0;
    IVR_CUDA(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
    if (g_dedup_timing && !g_dedup_ev[0])
        for (auto& ev : g_dedup_ev) IVR_CUDA(cudaEventCreate(&ev));
    if (g_dedup_timing) cudaEventRecord(g_dedup_ev[0], st);
    IVR_TRY(launch_banded(e_dev, n, 0, d, window, thr, mask_ws_dev, cos_prev_dev, sm_count, st));
    if (g_dedup_timing) { cudaEventRecord(g_dedup_ev[1], st); cudaEventRecord(g_dedup_ev[2], st); }
    IVR_CUDA(cudaMemsetAsync(keep_dev, 0, static_cast<size_t>(n), st));
    if (n_scenes > 0) {
        const int threads = 128;
        window_resolve_kernel<<<static_cast<unsigned>((n_scenes + threads - 1) / threads), threads, 0, st>>>(
            mask_ws_dev, scene_start_dev, scene_end_dev, n_scenes, n, window, keep_dev);
        IVR_CUDA(cudaGetLastError());
    }
    if (g_dedup_timing) { cudaEventRecord(g_dedup_ev[3], st); g_dedup_ev_valid = true; }
    return IVR_OK;
}

int dedup_chain_device(const float* e_dev, int64_t n, int d, const int64_t* scene_start_dev,
                       const int64_t* scene_end_dev, int64_t n_scenes, int min_distance, float thr,
                       int force_last, int fifo, uint8_t* keep_dev, cudaStream_t st) {
    if (n <= 0) return IVR_OK;
    IVR_CUDA(cudaMemsetAsync(keep_dev, 0, static_cast<size_t>(n), st));
    if (n_scenes <= 0) return IVR_OK;
    const int threads = 128;
    const int64_t blocks = (n_scenes * 32 + threads - 1) / threads;
    chain_resolve_kernel<<<static_cast<unsigned>(blocks), threads, 0, st>>>(
        e_dev, d, scene_start_dev, scene_end_dev, n_scenes, n, min_distance, thr, force_last, fifo, keep_dev);
    IVR_CUDA(cudaGetLastError());
    return IVR_OK;
}

}  // namespace ivr

// "Next" rows of the hot-path scope (SURVEY.md §8f): batched reference statistics and the streaming first-match
// gallery scan of the reference's face tracker.
//
//   ref_stats_batched_kernel   mean vector + max distance per class, all classes in one launch
//                              (similar_face_filtering/filter_faces_using_reference.py:85-99, once per class at :161-164)
//   first_match_stream_kernel  Net.check_if_face_exists + add_face
//                              (face_detection_and_extraction/face_extraction/extract_and_label_faces_from_dataset.py:101-121):
//                              for every query, in order: scan the gallery in ascending order, the FIRST entry with
//                              (dist < normal_thres and iou > 0.1) or dist < harsh_thres wins and is overwritten by the
//                              query (feature + bbox); otherwise the query is appended.  Queries depend on each other
//                              through the gallery, so one CTA walks them sequentially; each query's scan is parallel
//                              (one warp per gallery entry, 32 entries per round, early exit after the first hit).
#include <mutex>

#include "ffr_common.cuh"

namespace ffr {

namespace {

__global__ void __launch_bounds__(256)
ref_stats_batched_kernel(const float* __restrict__ x, const int32_t* __restrict__ offsets, int32_t dim,
                         float* __restrict__ mean, float* __restrict__ thres, int mode) {
    extern __shared__ __align__(16) float s_mean[];   // dim floats + 8 warp maxima
    float* s_max = s_mean + dim;
    const int c = blockIdx.x;
    const int32_t lo = offsets[c], hi = offsets[c + 1];
    const int32_t n = hi - lo;
    for (int d = threadIdx.x; d < dim; d += blockDim.x) {
        float acc = 0.f;
        for (int i = lo; i < hi; ++i) acc += x[static_cast<int64_t>(i) * dim + d];     // np.mean(axis=0): row order
        const float m = __fdiv_rn(acc, static_cast<float>(n));
        s_mean[d] = m;
        mean[static_cast<int64_t>(c) * dim + d] = m;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    float wmax = 0.f;
    for (int i = lo + warp; i < hi; i += nw)          // the distance K2s will compute for this row as a candidate, bit for bit
        wmax = fmaxf(wmax, k2s_euclid_dist(x + static_cast<int64_t>(i) * dim, s_mean, dim, lane, mode));
    if (lane == 0) s_max[warp] = wmax;
    __syncthreads();
    if (threadIdx.x == 0) {
        float m = 0.f;
        for (int w = 0; w < nw; ++w) m = fmaxf(m, s_max[w]);
        thres[c] = m;
    }
}

// modules/utils/image.py:124-143
__device__ __forceinline__ float bbox_iou(const float* a, const float* b) {
    const float xd = fminf(a[2], b[2]) - fmaxf(a[0], b[0]);
    const float yd = fminf(a[3], b[3]) - fmaxf(a[1], b[1]);
    if (xd < 0.f || yd < 0.f) return 0.f;
    const float inter = xd * yd;
    return inter / (((a[2] - a[0]) * (a[3] - a[1])) + ((b[2] - b[0]) * (b[3] - b[1])) - inter);
}

constexpr int kScanThreads = 256;
constexpr int kPasses = 4;                            // groups of four entries a warp scores side by side (independent chains)
constexpr int kScanPerWarp = 4 * kPasses;             // gallery entries per warp and round (eight lanes each): 128 entries per round
constexpr int kNone = 0x7FFFFFFF;
constexpr int kQueryDepth = 8;                        // queries in flight global -> shared (cp.async ring)

__device__ __forceinline__ void cp_async_f32(float* smem_dst, const float* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// The reference tracker (Net.check_if_face_exists + add_face, extract_and_label_faces_from_dataset.py:101-121) as ONE
// resident CTA: queries depend on each other through the gallery, so they are walked in order, and what there is to make
// fast is the latency of one query.  Round 2:
//   * kSmemGallery: the gallery (features + boxes) lives in shared memory for the whole launch when capacity x dim fits
//     (write-through to the global copy, which stays the state between launches); larger galleries are read through L1 / L2
//     (measured: 5-15 % slower per query -- a ~100-entry gallery stays L1-resident either way);
//   * the next kQueryDepth - 1 queries and their boxes are on their way global -> shared (cp.async ring) while the current one
//     is scanned (the first form loaded each query synchronously; a register-staged prefetch measured slower than the ring);
//   * EIGHT warps, 128 entries per round, EIGHT LANES per entry: a warp scores four groups of four entries side by side (16
//     independent accumulator chains, one query read per four gallery reads, three shuffle steps per sum), |q| is computed
//     once per query, ONE barrier per round and one per query.  ncu on an intermediate form (32 warps, four entries each): 242
//     warp-instructions per warp and query of which ~50 were arithmetic -- the loop was ISSUE-bound (59 % issue-active on all
//     four schedulers) on bookkeeping that every warp repeats; what is left at dim 512 is the SM's 128 B/cycle of shared
//     memory / L1 bandwidth (the whole gallery passes through it once per query).
//   Measured (tools/bench_tracker.py, 20 000 queries, ~110 gallery entries; first form -> this one): 128-d 2.05 -> 1.22 us per
//   query, 256-d 2.21 -> 1.64, 512-d 2.52 -> 2.54 (resident) / 2.59 -> 2.94 (capacity 4096: out of L1 / L2).
// The reference's formulas (:104 / :106) with IEEE sqrt / division; the order of the fp32 sums differs from NumPy's (as any
// order does) -- the reference's own (found, faceid) trajectories are reproduced (tests/golden/label_scan_ref.npz).
template <bool kSmemGallery, bool kEuclid>
__global__ void __launch_bounds__(kScanThreads, 1)
first_match_stream_kernel(float* __restrict__ g_feat, float* __restrict__ g_bbox, int32_t* __restrict__ g_count, int32_t cap,
                          const float* __restrict__ queries, const float* __restrict__ qboxes, int32_t n_queries,
                          int32_t dim, int metric, float normal_thres, float harsh_thres, int32_t* __restrict__ match_idx) {
    extern __shared__ float s_mem[];                  // [kQueryDepth][dim] queries | [kQueryDepth][4] boxes | kSmemGallery: [cap][dim] + [cap][4]
    __shared__ int s_first[2][2];
    __shared__ float s_qn[2];                         // |q| of the current / next query (cosine)
    float* s_q = s_mem;
    float* s_qb = s_mem + kQueryDepth * dim;
    float* s_gf = s_qb + kQueryDepth * 4;
    float* s_gb = s_gf + static_cast<size_t>(kSmemGallery ? cap : 0) * dim;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = kScanThreads / 32;
    const bool vec = (dim & 31) == 0;
    int count = *g_count;
    if (kSmemGallery) {
        for (int64_t i = threadIdx.x; i < static_cast<int64_t>(count) * dim; i += kScanThreads) s_gf[i] = g_feat[i];
        for (int i = threadIdx.x; i < count * 4; i += kScanThreads) s_gb[i] = g_bbox[i];
    }
    const float* gf_base = kSmemGallery ? s_gf : g_feat;
    const float* gb_base = kSmemGallery ? s_gb : g_bbox;
    // one cp.async group per query (committed by every thread, empty past the end): group q is complete once at most
    // kQueryDepth - 2 younger groups are pending
    auto fetch_query = [&](int q) {
        if (q < n_queries) {
            const int buf = q % kQueryDepth;
            const float* qf = queries + static_cast<int64_t>(q) * dim;
            for (int d = threadIdx.x; d < dim; d += kScanThreads) cp_async_f32(s_q + buf * dim + d, qf + d);
            if (qboxes != nullptr && threadIdx.x < 4) cp_async_f32(s_qb + buf * 4 + threadIdx.x, qboxes + static_cast<int64_t>(q) * 4 + threadIdx.x);
        }
        cp_async_commit();
    };
    for (int q = 0; q < kQueryDepth - 1; ++q) fetch_query(q);
    if (threadIdx.x < 4) (&s_first[0][0])[threadIdx.x] = kNone;
    cp_async_wait_group<kQueryDepth - 3>();           // queries 0 AND 1 (the loop keeps one more group complete than it consumes)
    __syncthreads();
    if (warp == 0 && !kEuclid) {
        float a = 0.f;
        for (int d = lane; d < dim; d += 32) a = fmaf(s_q[d], s_q[d], a);
        a = warp_sum(a);
        if (lane == 0) s_qn[0] = __fsqrt_rn(a);
    }
    __syncthreads();
    for (int q = 0; q < n_queries; ++q) {
        const int cur = q & 1, qbuf = q % kQueryDepth;
        if (threadIdx.x < 2) s_first[cur ^ 1][threadIdx.x] = kNone;   // last read before the barrier that ended query q - 1
        const float* sq = s_q + qbuf * dim;
        fetch_query(q + kQueryDepth - 1);                             // into the buffer query q - 1 has just left
        const float qnorm = s_qn[cur];
        // |q| of the NEXT query, once, by the last warp (its group landed before the barrier that ended query q - 1)
        if (warp == nw - 1 && q + 1 < n_queries && !kEuclid) {
            const float* sn = s_q + ((q + 1) % kQueryDepth) * dim;
            float a = 0.f;
            for (int d = lane; d < dim; d += 32) a = fmaf(sn[d], sn[d], a);
            a = warp_sum(a);
            if (lane == 0) s_qn[cur ^ 1] = __fsqrt_rn(a);
        }
        int first = kNone;
        int slot = 0;                                  // both slots of this parity are kNone at the top of the query
        for (int base = 0; base < count; base += nw * kScanPerWarp) {
            // EIGHT lanes per entry, four entries per warp side by side: lane = 8 * j + k scores entry base + 4 * warp + j over
            // the elements d = k, k + 8, ... (float4 steps when dim % 32 == 0), three shuffle steps finish the sums, lane 8 j
            // applies the rule.  (Warp per entry -- the first form -- is a ~500-cycle dependent chain per entry and 10 shuffles
            // per warp and entry: with 32 warps it kept the SM's shuffle and LDS pipes busy for ~2 us per query whatever the
            // gallery size.)
            const int j = lane >> 3, k = lane & 7;
            int i[kPasses];
            const float* gf[kPasses];
            float a[kPasses], b[kPasses];
#pragma unroll
            for (int ps = 0; ps < kPasses; ++ps) {
                i[ps] = base + warp * kScanPerWarp + ps * 4 + j;
                gf[ps] = gf_base + static_cast<int64_t>(i[ps] < count ? i[ps] : 0) * dim;
                a[ps] = 0.f;
                b[ps] = 0.f;
            }
            if (vec) {
                const float4* q4 = reinterpret_cast<const float4*>(sq);
                for (int d = k; d < (dim >> 2); d += 8) {
                    const float4 qv = q4[d];
#pragma unroll
                    for (int ps = 0; ps < kPasses; ++ps) {
                        const float4 gv = reinterpret_cast<const float4*>(gf[ps])[d];
                        if (kEuclid) {
                            float t = gv.x - qv.x; a[ps] = fmaf(t, t, a[ps]);
                            t = gv.y - qv.y; a[ps] = fmaf(t, t, a[ps]);
                            t = gv.z - qv.z; a[ps] = fmaf(t, t, a[ps]);
                            t = gv.w - qv.w; a[ps] = fmaf(t, t, a[ps]);
                        } else {
                            a[ps] = fmaf(gv.x, qv.x, a[ps]); a[ps] = fmaf(gv.y, qv.y, a[ps]); a[ps] = fmaf(gv.z, qv.z, a[ps]); a[ps] = fmaf(gv.w, qv.w, a[ps]);
                            b[ps] = fmaf(gv.x, gv.x, b[ps]); b[ps] = fmaf(gv.y, gv.y, b[ps]); b[ps] = fmaf(gv.z, gv.z, b[ps]); b[ps] = fmaf(gv.w, gv.w, b[ps]);
                        }
                    }
                }
            } else {
                for (int d = k; d < dim; d += 8) {
                    const float qv = sq[d];
#pragma unroll
                    for (int ps = 0; ps < kPasses; ++ps) {
                        const float gv = gf[ps][d];
                        if (kEuclid) { const float t = gv - qv; a[ps] = fmaf(t, t, a[ps]); }
                        else         { a[ps] = fmaf(gv, qv, a[ps]); b[ps] = fmaf(gv, gv, b[ps]); }
                    }
                }
            }
#pragma unroll
            for (int o = 4; o > 0; o >>= 1)
#pragma unroll
                for (int ps = 0; ps < kPasses; ++ps) {
                    a[ps] += __shfl_xor_sync(0xffffffffu, a[ps], o);
                    if (!kEuclid) b[ps] += __shfl_xor_sync(0xffffffffu, b[ps], o);
                }
            // lane 8 j finishes entry j of the first pass, lane 8 j + 1 (which holds the same sums) entry j of the second
            if (k < kPasses) {
                int ii = i[0];
                float aa = a[0], bb = b[0];
#pragma unroll
                for (int ps = 1; ps < kPasses; ++ps) { ii = k == ps ? i[ps] : ii; aa = k == ps ? a[ps] : aa; bb = k == ps ? b[ps] : bb; }
                if (ii < count) {
                    const float dist = kEuclid ? __fsqrt_rn(aa)                                                 // :104
                                               : 1.f - __fdiv_rn(aa, __fmul_rn(__fsqrt_rn(bb), qnorm));         // :106
                    const float iou = qboxes != nullptr ? bbox_iou(gb_base + static_cast<int64_t>(ii) * 4, s_qb + qbuf * 4) : 0.f;
                    if ((dist < normal_thres && iou > 0.1f) || dist < harsh_thres) atomicMin(&s_first[cur][slot], ii);   // :110
                }
            }
            __syncthreads();
            first = s_first[cur][slot];
            if (first != kNone) break;                 // every entry below base + 128 has been examined
            slot ^= 1;
        }
        int dst;
        if (first != kNone) {                          // :113-114 overwrite the matched entry
            dst = first;
            if (threadIdx.x == 0) match_idx[q] = first;
        } else if (count < cap) {                      // add_face :118-121
            dst = count;
            if (threadIdx.x == 0) match_idx[q] = -1 - count;
            ++count;
        } else {
            dst = -1;
            if (threadIdx.x == 0) match_idx[q] = INT32_MIN;    // gallery full: query dropped
        }
        if (dst >= 0) {
            for (int d = threadIdx.x; d < dim; d += kScanThreads) {
                const float v = sq[d];
                g_feat[static_cast<int64_t>(dst) * dim + d] = v;
                if (kSmemGallery) s_gf[static_cast<int64_t>(dst) * dim + d] = v;
            }
            if (threadIdx.x < 4 && qboxes != nullptr) {
                const float v = s_qb[qbuf * 4 + threadIdx.x];
                g_bbox[static_cast<int64_t>(dst) * 4 + threadIdx.x] = v;
                if (kSmemGallery) s_gb[dst * 4 + threadIdx.x] = v;
            }
        }
        cp_async_wait_group<kQueryDepth - 3>();        // queries q + 1 and q + 2 have landed
        __syncthreads();                               // ... gallery row written, |q + 1| published, this query's slots read by everyone
    }
    if (threadIdx.x == 0) *g_count = count;
}

}  // namespace

int launch_ref_stats_batched(const float* ref_feat, const int32_t* offsets, int32_t n_classes, int32_t dim, float* mean,
                             float* thres, cudaStream_t s) {
    if (n_classes == 0) return FFR_OK;
    const size_t smem = (static_cast<size_t>(dim) + 8) * sizeof(float);
    ref_stats_batched_kernel<<<static_cast<unsigned>(n_classes), 256, smem, s>>>(ref_feat, offsets, dim, mean, thres,
                                                                                    k2s_form(ref_feat, ref_feat, 1, dim));
    FFR_LAUNCH_CHECK("ref_stats_batched");
    return FFR_OK;
}

int launch_first_match_stream(float* g_feat, float* g_bbox, int32_t* g_count, int32_t cap, const float* queries,
                              const float* qboxes, int32_t n_queries, int32_t dim, int metric, float normal_thres,
                              float harsh_thres, int32_t* match_idx, cudaStream_t s) {
    if (n_queries == 0) return FFR_OK;
    const size_t q_bytes = static_cast<size_t>(kQueryDepth) * (static_cast<size_t>(dim) + 4) * sizeof(float);
    const size_t g_bytes = static_cast<size_t>(cap) * (static_cast<size_t>(dim) + 4) * sizeof(float);
    const bool in_smem = q_bytes + g_bytes <= 200 * 1024;      // e.g. 384 faces x 128-d, 96 x 512-d; larger galleries stay in L2
    {   // per-DEVICE function attribute: once for every device this process uses
        static std::mutex mu;
        static bool attr_set[kMaxDevices] = {};
        const int slot = current_device_slot();
        std::lock_guard<std::mutex> lock(mu);
        if (!attr_set[slot]) {
            FFR_CUDA_TRY(cudaFuncSetAttribute(first_match_stream_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024 + 64));
            FFR_CUDA_TRY(cudaFuncSetAttribute(first_match_stream_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024 + 64));
            FFR_CUDA_TRY(cudaFuncSetAttribute(first_match_stream_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024 + 64));
            FFR_CUDA_TRY(cudaFuncSetAttribute(first_match_stream_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024 + 64));
            attr_set[slot] = true;
        }
    }
    if (q_bytes > 200 * 1024) { set_error("first_match_stream: dim %d too large", dim); return FFR_ERR_UNSUPPORTED; }
    auto launch = [&](auto kern, size_t smem) {
        kern<<<1, kScanThreads, smem, s>>>(g_feat, g_bbox, g_count, cap, queries, qboxes, n_queries, dim, metric, normal_thres, harsh_thres,
                                           match_idx);
    };
    const bool euclid = metric == FFR_METRIC_EUCLID;
    if (in_smem) { if (euclid) launch(first_match_stream_kernel<true, true>, q_bytes + g_bytes); else launch(first_match_stream_kernel<true, false>, q_bytes + g_bytes); }
    else         { if (euclid) launch(first_match_stream_kernel<false, true>, q_bytes); else launch(first_match_stream_kernel<false, false>, q_bytes); }
    FFR_LAUNCH_CHECK("first_match_stream");
    return FFR_OK;
}

}  // namespace ffr

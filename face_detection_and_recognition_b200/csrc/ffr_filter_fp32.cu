// K2s -- exact fp32 CUDA-core filter (streaming, small reference sets) + K5 reference statistics.
//
// Replaces the reference's per-row test
//     similar_face_filtering/filter_faces_using_reference.py:186-189   np.linalg.norm(out - mu) <= thres
// (metric euclid, n_ref = 1, ref = the class mean vector) and the per-pair expressions of
//     face_detection_and_extraction/face_extraction/extract_and_label_faces_from_dataset.py:104 (euclid)
//     .../extract_and_label_faces_from_dataset.py:106  1 - inner/(|f||g|)                    (cosine)
// for reference sets too small to feed the tensor cores (the HBM-bound regime: 4*dim bytes read per
// candidate, 9 bytes written), and serves as the exact path for the euclid metric at any n_ref.
// Arithmetic is fp32 throughout with direct differences for euclid (same cancellation behaviour as
// NumPy's (out - mu) then dot) and true IEEE sqrt/div.
//
// One warp owns a candidate row: lane l holds float4 #(l + 32 j) of the row in registers (coalesced,
// streaming loads), walks the reference rows (registers when the whole reference set fits in 8 float4
// per lane -- always true for the reference's n_ref = 1 -- else L1/L2-resident global loads), reduces
// each score with warp shuffles, and keeps a running best with strict comparison in ascending index
// order, which is np.argmax / np.argmin first-occurrence.
#include <stdlib.h>

#include "ffr_common.cuh"

namespace ffr {

namespace {

constexpr int kThreads = 256;

template <int NV, bool kCosine>
__device__ __forceinline__ void score_row(const float4 (&c)[NV], const float4 (&r)[NV], float cc_sqrt, float& score) {
    // returns cosine similarity or euclid distance of the candidate (regs c) and one reference (regs r)
    float a = 0.f, b = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        if (kCosine) {
            a = fmaf(c[j].x, r[j].x, a); a = fmaf(c[j].y, r[j].y, a);
            a = fmaf(c[j].z, r[j].z, a); a = fmaf(c[j].w, r[j].w, a);
            b = fmaf(r[j].x, r[j].x, b); b = fmaf(r[j].y, r[j].y, b);
            b = fmaf(r[j].z, r[j].z, b); b = fmaf(r[j].w, r[j].w, b);
        } else {
            float d;
            d = c[j].x - r[j].x; a = fmaf(d, d, a);
            d = c[j].y - r[j].y; a = fmaf(d, d, a);
            d = c[j].z - r[j].z; a = fmaf(d, d, a);
            d = c[j].w - r[j].w; a = fmaf(d, d, a);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        if (kCosine) b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (kCosine) score = __fdiv_rn(a, __fmul_rn(__fsqrt_rn(b), cc_sqrt));   // inner / (|r| * |c|)   (:106)
    else         score = __fsqrt_rn(a);                                      // |c - r|               (:189, :104)
}

template <int NV>
__device__ __forceinline__ void load_row(const float* __restrict__ base, int32_t dim, int lane, float4 (&v)[NV],
                                         bool streaming) {
    const float4* p = reinterpret_cast<const float4*>(base);
    const int nvec = dim >> 2;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int k = lane + 32 * j;
        if (k < nvec) v[j] = streaming ? ldg_stream_f4(p + k) : __ldg(p + k);
        else          v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// kSelf (ffr_filter_self, kRegRefs 0): cand = rows [self.row0, ...) of ref; candidate row g skips reference g
// (FFR_SELF_OTHERS) or every reference >= g (FFR_SELF_EARLIER); a row with none left gets index -1 and -inf / +inf
template <int NV, bool kCosine, int kRegRefs, bool kSelf = false>
__global__ void __launch_bounds__(kThreads)
filter_fp32_kernel(const float* __restrict__ ref, int64_t n_ref, const float* __restrict__ cand, int64_t n_cand,
                   int32_t dim, float thr, int64_t ref_index_base,
                   uint8_t* __restrict__ keep, int32_t* __restrict__ best_idx, float* __restrict__ best_val,
                   Band band, SelfArgs self) {
    static_assert(!kSelf || kRegRefs == 0, "self form: references from global memory");
    const int lane = threadIdx.x & 31;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;

    float4 rreg[kRegRefs > 0 ? kRegRefs : 1][NV];
    if (kRegRefs > 0) {
#pragma unroll
        for (int i = 0; i < kRegRefs; ++i)
            if (i < n_ref) load_row<NV>(ref + static_cast<int64_t>(i) * dim, dim, lane, rreg[i], false);
    }

    // kRowsInFlight candidate rows are loaded before any is consumed, so that every warp keeps several
    // independent 512-byte requests outstanding (HBM latency x bandwidth needs ~40 KB in flight per SM)
    constexpr int kRowsInFlight = (NV <= 2) ? 4 : 2;
    for (int64_t row0 = warp * kRowsInFlight; row0 < n_cand; row0 += nwarps * kRowsInFlight) {
      float4 cbuf[kRowsInFlight][NV];
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u)
        if (row0 + u < n_cand) load_row<NV>(cand + (row0 + u) * dim, dim, lane, cbuf[u], true);
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {
        const int64_t row = row0 + u;
        if (row >= n_cand) break;
        float4 (&c)[NV] = cbuf[u];
        float cc_sqrt = 0.f;
        if (kCosine) {
            float cc = 0.f;
#pragma unroll
            for (int j = 0; j < NV; ++j) {
                cc = fmaf(c[j].x, c[j].x, cc); cc = fmaf(c[j].y, c[j].y, cc);
                cc = fmaf(c[j].z, c[j].z, cc); cc = fmaf(c[j].w, c[j].w, cc);
            }
            cc_sqrt = __fsqrt_rn(warp_sum(cc));
        }
        float best = kCosine ? -INFINITY : INFINITY;
        int32_t bi = kSelf ? -1 : 0;
        if (kRegRefs > 0) {
#pragma unroll
            for (int i = 0; i < kRegRefs; ++i) {
                if (i < n_ref) {
                    float s;
                    score_row<NV, kCosine>(c, rreg[i], cc_sqrt, s);
                    const bool better = kCosine ? (s > best) : (s < best);
                    if (better || i == 0) { best = s; bi = i; }
                }
            }
        } else {
            const int64_t g = self.row0 + row;
            const int64_t i_end = kSelf && self.mode == FFR_SELF_EARLIER ? g : n_ref;
            for (int64_t i = 0; i < i_end; ++i) {
                if (kSelf && i == g) continue;
                float4 r[NV];
                load_row<NV>(ref + i * dim, dim, lane, r, false);
                float s;
                score_row<NV, kCosine>(c, r, cc_sqrt, s);
                const bool better = kCosine ? (s > best) : (s < best);
                if (better || (kSelf ? bi < 0 : i == 0)) { best = s; bi = static_cast<int32_t>(i); }
            }
        }
        if (lane == 0) {
            const bool k = (kCosine ? (best >= thr) : (best <= thr)) && (!kSelf || bi >= 0);
            keep[row] = k ? 1 : 0;
            best_idx[row] = static_cast<int32_t>(bi + ref_index_base);
            if (best_val != nullptr) best_val[row] = best;
            if (band.count != nullptr && fabsf(best - thr) <= band.tol) {
                const int32_t slot = atomicAdd(band.count, 1);
                if (band.rows != nullptr && slot < band.cap) band.rows[slot] = row;
            }
        }
      }
    }
}

// Short rows (dim 128 / 256) against one or two references -- the reference's literal mode (one mean vector): a candidate
// row is owned by L = dim / 16 lanes (4 float4 each), so a warp instruction covers 32 / L rows and a score needs log2(L)
// shuffles instead of five.  The warp-per-row kernel above is issue bound at ~84 % of the HBM copy rate for 128-d rows;
// here the same bytes cost a third of the instructions.  Same per-pair formulas; the references (and |r|) live in
// registers.
template <int L, bool kCosine>
__global__ void __launch_bounds__(kThreads)
filter_fp32_sub_kernel(const float* __restrict__ ref, int32_t n_ref, const float* __restrict__ cand, int64_t n_cand,
                       int32_t dim, float thr, int64_t ref_index_base,
                       uint8_t* __restrict__ keep, int32_t* __restrict__ best_idx, float* __restrict__ best_val,
                       Band band) {
    constexpr int kRowsPerWarp = 32 / L;
    constexpr int kGroups = 2;                                      // row groups in flight per warp (4 KB)
    const int lane = threadIdx.x & 31, sub = lane % L, rsel = lane / L;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;
    float4 rr[2][4];
    float r_sqrt[2] = {0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        float b = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            rr[i][j] = (i < n_ref) ? __ldg(reinterpret_cast<const float4*>(ref + static_cast<int64_t>(i) * dim) + sub + L * j)
                                   : make_float4(0.f, 0.f, 0.f, 0.f);
            b = fmaf(rr[i][j].x, rr[i][j].x, b); b = fmaf(rr[i][j].y, rr[i][j].y, b);
            b = fmaf(rr[i][j].z, rr[i][j].z, b); b = fmaf(rr[i][j].w, rr[i][j].w, b);
        }
#pragma unroll
        for (int o = L / 2; o > 0; o >>= 1) b += __shfl_xor_sync(0xffffffffu, b, o);
        r_sqrt[i] = __fsqrt_rn(b);
    }
    for (int64_t r0 = warp * (kGroups * kRowsPerWarp); r0 < n_cand; r0 += nwarps * (kGroups * kRowsPerWarp)) {
        float4 c[kGroups][4];
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const int64_t row = r0 + g * kRowsPerWarp + rsel;
            const float4* p = reinterpret_cast<const float4*>(cand + (row < n_cand ? row : n_cand - 1) * dim);
#pragma unroll
            for (int j = 0; j < 4; ++j) c[g][j] = ldg_stream_f4(p + sub + L * j);
        }
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const int64_t row = r0 + g * kRowsPerWarp + rsel;
            float cc_sqrt = 0.f;
            if (kCosine) {
                float cc = 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    cc = fmaf(c[g][j].x, c[g][j].x, cc); cc = fmaf(c[g][j].y, c[g][j].y, cc);
                    cc = fmaf(c[g][j].z, c[g][j].z, cc); cc = fmaf(c[g][j].w, c[g][j].w, cc);
                }
#pragma unroll
                for (int o = L / 2; o > 0; o >>= 1) cc += __shfl_xor_sync(0xffffffffu, cc, o);
                cc_sqrt = __fsqrt_rn(cc);
            }
            float best = kCosine ? -INFINITY : INFINITY;
            int32_t bi = 0;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if (i < n_ref) {
                    float a = 0.f;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (kCosine) {
                            a = fmaf(c[g][j].x, rr[i][j].x, a); a = fmaf(c[g][j].y, rr[i][j].y, a);
                            a = fmaf(c[g][j].z, rr[i][j].z, a); a = fmaf(c[g][j].w, rr[i][j].w, a);
                        } else {
                            float d;
                            d = c[g][j].x - rr[i][j].x; a = fmaf(d, d, a);
                            d = c[g][j].y - rr[i][j].y; a = fmaf(d, d, a);
                            d = c[g][j].z - rr[i][j].z; a = fmaf(d, d, a);
                            d = c[g][j].w - rr[i][j].w; a = fmaf(d, d, a);
                        }
                    }
#pragma unroll
                    for (int o = L / 2; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
                    const float sc = kCosine ? __fdiv_rn(a, __fmul_rn(r_sqrt[i], cc_sqrt)) : __fsqrt_rn(a);
                    const bool better = kCosine ? (sc > best) : (sc < best);
                    if (better || i == 0) { best = sc; bi = i; }
                }
            }
            if (sub == 0 && row < n_cand) {
                const bool k = kCosine ? (best >= thr) : (best <= thr);
                keep[row] = k ? 1 : 0;
                best_idx[row] = static_cast<int32_t>(bi + ref_index_base);
                if (best_val != nullptr) best_val[row] = best;
                if (band.count != nullptr && fabsf(best - thr) <= band.tol) {
                    const int32_t slot = atomicAdd(band.count, 1);
                    if (band.rows != nullptr && slot < band.cap) band.rows[slot] = row;
                }
            }
        }
    }
}

// catch-all: any dim / alignment; one warp per candidate, scalar loads (kSelf: as filter_fp32_kernel)
template <bool kCosine, bool kSelf = false>
__global__ void __launch_bounds__(kThreads)
filter_fp32_generic_kernel(const float* __restrict__ ref, int64_t n_ref, const float* __restrict__ cand,
                           int64_t n_cand, int32_t dim, float thr, int64_t ref_index_base,
                           uint8_t* __restrict__ keep, int32_t* __restrict__ best_idx, float* __restrict__ best_val,
                           Band band, SelfArgs self) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;
    for (int64_t row = warp; row < n_cand; row += nwarps) {
        const float* c = cand + row * dim;
        float cc_sqrt = 0.f;
        if (kCosine) {
            float cc = 0.f;
            for (int k = lane; k < dim; k += 32) { const float t = __ldg(c + k); cc = fmaf(t, t, cc); }
            cc_sqrt = __fsqrt_rn(warp_sum(cc));
        }
        float best = kCosine ? -INFINITY : INFINITY;
        int32_t bi = kSelf ? -1 : 0;
        const int64_t g = self.row0 + row;
        const int64_t i_end = kSelf && self.mode == FFR_SELF_EARLIER ? g : n_ref;
        for (int64_t i = 0; i < i_end; ++i) {
            if (kSelf && i == g) continue;
            const float* r = ref + i * dim;
            float a = 0.f, b = 0.f;
            for (int k = lane; k < dim; k += 32) {
                const float cv = __ldg(c + k), rv = __ldg(r + k);
                if (kCosine) { a = fmaf(cv, rv, a); b = fmaf(rv, rv, b); }
                else { const float d = cv - rv; a = fmaf(d, d, a); }
            }
            a = warp_sum(a);
            float s;
            if (kCosine) { b = warp_sum(b); s = __fdiv_rn(a, __fmul_rn(__fsqrt_rn(b), cc_sqrt)); }
            else s = __fsqrt_rn(a);
            const bool better = kCosine ? (s > best) : (s < best);
            if (better || (kSelf ? bi < 0 : i == 0)) { best = s; bi = static_cast<int32_t>(i); }
        }
        if (lane == 0) {
            const bool k = (kCosine ? (best >= thr) : (best <= thr)) && (!kSelf || bi >= 0);
            keep[row] = k ? 1 : 0;
            best_idx[row] = static_cast<int32_t>(bi + ref_index_base);
            if (best_val != nullptr) best_val[row] = best;
            if (band.count != nullptr && fabsf(best - thr) <= band.tol) {
                const int32_t slot = atomicAdd(band.count, 1);
                if (band.rows != nullptr && slot < band.cap) band.rows[slot] = row;
            }
        }
    }
}

// K5: mean vector + max distance from the mean (filter_faces_using_reference.py:85-99). One CTA.
//   mean[d] = (sum_i x[i,d]) / n   (np.mean over axis 0: sequential fp32 accumulation for n <= 8 rows per
//   pairwise block is not reproduced bit-for-bit; tolerance documented in the tests)
__global__ void __launch_bounds__(256)
ref_stats_kernel(const float* __restrict__ x, int32_t n, int32_t dim, float* __restrict__ mean, float* __restrict__ thres, int mode) {
    extern __shared__ __align__(16) float s_mean[];   // dim floats + 8 warp maxima
    float* s_max = s_mean + dim;
    for (int d = threadIdx.x; d < dim; d += blockDim.x) {
        float acc = 0.f;
        for (int i = 0; i < n; ++i) acc += x[static_cast<int64_t>(i) * dim + d];
        const float m = __fdiv_rn(acc, static_cast<float>(n));
        s_mean[d] = m;
        mean[d] = m;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    float wmax = 0.f;
    for (int i = warp; i < n; i += nw)                // the distance K2s will compute for this row as a candidate, bit for bit
        wmax = fmaxf(wmax, k2s_euclid_dist(x + static_cast<int64_t>(i) * dim, s_mean, dim, lane, mode));
    if (lane == 0) s_max[warp] = wmax;
    __syncthreads();
    if (threadIdx.x == 0) {
        float m = 0.f;
        for (int w = 0; w < nw; ++w) m = fmaxf(m, s_max[w]);
        *thres = m;
    }
}

// Value pass of the tcgen05 Euclid filter: K2 + K3 chose best_idx; the distance to that reference is recomputed here with
// exactly the arithmetic K2s uses for the same (row, reference) pair (k2s_euclid_dist in K2s's mode for n_ref > 2), so keep and
// best_val are bit-identical to the FFR_FLAG_FORCE_FP32 result wherever the index agrees.  One warp per row; HBM-bound (one
// read of the candidate matrix, the winners' rows mostly from L2).
// kSelf: a row without an eligible reference (best_idx -1) gets keep 0 and +inf, and never enters the band
template <int kMode, bool kSelf = false>
__global__ void __launch_bounds__(kThreads)
euclid_value_kernel(const float* __restrict__ ref, const float* __restrict__ cand, int64_t n_cand, int32_t dim, float thr,
                    int64_t ref_index_base, uint8_t* __restrict__ keep, const int32_t* __restrict__ best_idx,
                    float* __restrict__ best_val, Band band) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;
    for (int64_t row = warp; row < n_cand; row += nwarps) {
        const int64_t ri = static_cast<int64_t>(__ldg(best_idx + row)) - ref_index_base;
        if constexpr (kSelf) {
            if (ri < 0) {
                if (lane == 0) { keep[row] = 0; if (best_val != nullptr) best_val[row] = INFINITY; }
                continue;
            }
        }
        const float d = k2s_euclid_dist(cand + row * dim, ref + ri * dim, dim, lane, kMode);
        if (lane == 0) {
            keep[row] = d <= thr ? 1 : 0;
            if (best_val != nullptr) best_val[row] = d;
            if (band.count != nullptr && fabsf(d - thr) <= band.tol) {
                const int32_t slot = atomicAdd(band.count, 1);
                if (band.rows != nullptr && slot < band.cap) band.rows[slot] = row;
            }
        }
    }
}

template <int NV, bool kCosine>
int launch_vec(const float* ref, int64_t n_ref, const float* cand, int64_t n_cand, int32_t dim, float thr,
               int64_t base, const FilterOut& o, dim3 g, cudaStream_t s) {
    const dim3 b(kThreads);
    const int64_t ref_vecs = n_ref * NV;
    if (ref_vecs <= 8) {
        if (n_ref == 1)      filter_fp32_kernel<NV, kCosine, 1><<<g, b, 0, s>>>(ref, n_ref, cand, n_cand, dim, thr, base, o.keep, o.idx, o.val, o.band, kNoSelf);
        else if (n_ref == 2) filter_fp32_kernel<NV, kCosine, 2><<<g, b, 0, s>>>(ref, n_ref, cand, n_cand, dim, thr, base, o.keep, o.idx, o.val, o.band, kNoSelf);
        else if (n_ref <= 4) filter_fp32_kernel<NV, kCosine, (NV <= 2 ? 4 : 1)><<<g, b, 0, s>>>(ref, n_ref, cand, n_cand, dim, thr, base, o.keep, o.idx, o.val, o.band, kNoSelf);
        else                 filter_fp32_kernel<NV, kCosine, (NV == 1 ? 8 : 1)><<<g, b, 0, s>>>(ref, n_ref, cand, n_cand, dim, thr, base, o.keep, o.idx, o.val, o.band, kNoSelf);
    } else {
        filter_fp32_kernel<NV, kCosine, 0><<<g, b, 0, s>>>(ref, n_ref, cand, n_cand, dim, thr, base, o.keep, o.idx, o.val, o.band, kNoSelf);
    }
    FFR_LAUNCH_CHECK("filter_fp32");
    return FFR_OK;
}

}  // namespace

int k2s_form(const float* ref, const float* cand, int64_t n_ref, int32_t dim) {
    const bool vec_ok = (dim % 4 == 0) && dim <= 1024 && ((reinterpret_cast<uintptr_t>(ref) & 15) == 0) &&
                        ((reinterpret_cast<uintptr_t>(cand) & 15) == 0);
    if (!vec_ok) return 0;                                                     // filter_fp32_generic_kernel
    if (n_ref <= 2 && (dim == 128 || dim == 256)) return dim == 128 ? 16 : 32;   // filter_fp32_sub_kernel<dim / 16>
    const int nv = (dim + 127) / 128;                                          // filter_fp32_kernel<NV>
    return nv <= 1 ? 1 : (nv <= 2 ? 2 : (nv <= 4 ? 4 : 8));
}

int launch_filter_fp32(const float* ref, int64_t n_ref, const float* cand, int64_t n_cand, int32_t dim, int metric,
                       float thr, int64_t ref_index_base, const FilterOut& o, cudaStream_t s) {
    if (n_cand == 0) return FFR_OK;
    const int sms = num_sms();
    const int64_t blocks_needed = (n_cand + (kThreads / 32) - 1) / (kThreads / 32);
    int64_t grid = blocks_needed < static_cast<int64_t>(sms) * 8 ? blocks_needed : static_cast<int64_t>(sms) * 8;
    const dim3 g(static_cast<unsigned>(grid));
    const bool cosine = metric == FFR_METRIC_COSINE;
    const int form = k2s_form(ref, cand, n_ref, dim);
    if (form == 0) {
        if (cosine) filter_fp32_generic_kernel<true><<<g, kThreads, 0, s>>>(ref, n_ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band, kNoSelf);
        else        filter_fp32_generic_kernel<false><<<g, kThreads, 0, s>>>(ref, n_ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band, kNoSelf);
        FFR_LAUNCH_CHECK("filter_fp32_generic");
        return FFR_OK;
    }
    if (form >= 16) {
        const int64_t rows_per_warp = (dim == 128 ? 4 : 2) * 2;
        const int64_t w_needed = (n_cand + rows_per_warp - 1) / rows_per_warp;
        int64_t gsub = (w_needed + (kThreads / 32) - 1) / (kThreads / 32);
        if (gsub > static_cast<int64_t>(sms) * 8) gsub = static_cast<int64_t>(sms) * 8;
        const dim3 gs(static_cast<unsigned>(gsub));
        const int32_t nr = static_cast<int32_t>(n_ref);
        if (dim == 128) {
            if (cosine) filter_fp32_sub_kernel<8, true><<<gs, kThreads, 0, s>>>(ref, nr, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band);
            else        filter_fp32_sub_kernel<8, false><<<gs, kThreads, 0, s>>>(ref, nr, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band);
        } else {
            if (cosine) filter_fp32_sub_kernel<16, true><<<gs, kThreads, 0, s>>>(ref, nr, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band);
            else        filter_fp32_sub_kernel<16, false><<<gs, kThreads, 0, s>>>(ref, nr, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band);
        }
        FFR_LAUNCH_CHECK("filter_fp32_sub");
        return FFR_OK;
    }
#define FFR_DISPATCH(NV)                                                                                          \
    return cosine ? launch_vec<NV, true>(ref, n_ref, cand, n_cand, dim, thr, ref_index_base, o, g, s)             \
                  : launch_vec<NV, false>(ref, n_ref, cand, n_cand, dim, thr, ref_index_base, o, g, s)
    switch (form) {
        case 1: FFR_DISPATCH(1);
        case 2: FFR_DISPATCH(2);
        case 4: FFR_DISPATCH(4);
        default: FFR_DISPATCH(8);
    }
#undef FFR_DISPATCH
}

int launch_euclid_values(const float* ref, const float* cand, int64_t n_cand, int32_t dim, float thr, int64_t ref_index_base,
                         const FilterOut& o, int mode, cudaStream_t s, bool self) {
    if (n_cand == 0) return FFR_OK;
    int64_t grid = (n_cand + (kThreads / 32) - 1) / (kThreads / 32);
    if (grid > static_cast<int64_t>(num_sms()) * 8) grid = static_cast<int64_t>(num_sms()) * 8;
    const dim3 g(static_cast<unsigned>(grid));
    if (self) {
        switch (mode) {
            case 1: euclid_value_kernel<1, true><<<g, kThreads, 0, s>>>(ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band); break;
            case 2: euclid_value_kernel<2, true><<<g, kThreads, 0, s>>>(ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band); break;
            case 4: euclid_value_kernel<4, true><<<g, kThreads, 0, s>>>(ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band); break;
            case 8: euclid_value_kernel<8, true><<<g, kThreads, 0, s>>>(ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band); break;
            default: euclid_value_kernel<0, true><<<g, kThreads, 0, s>>>(ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band); break;
        }
        FFR_LAUNCH_CHECK("euclid_values");
        return FFR_OK;
    }
    switch (mode) {
        case 1: euclid_value_kernel<1><<<g, kThreads, 0, s>>>(ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band); break;
        case 2: euclid_value_kernel<2><<<g, kThreads, 0, s>>>(ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band); break;
        case 4: euclid_value_kernel<4><<<g, kThreads, 0, s>>>(ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band); break;
        case 8: euclid_value_kernel<8><<<g, kThreads, 0, s>>>(ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band); break;
        default: euclid_value_kernel<0><<<g, kThreads, 0, s>>>(ref, cand, n_cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, o.band); break;
    }
    FFR_LAUNCH_CHECK("euclid_values");
    return FFR_OK;
}

int launch_filter_fp32_self(const float* x, int64_t n, int64_t n_cand, int32_t dim, int metric, SelfArgs self, float thr,
                            const FilterOut& o, cudaStream_t s) {
    if (n_cand == 0) return FFR_OK;
    const float* cand = x + self.row0 * dim;
    const int sms = num_sms();
    const int64_t blocks_needed = (n_cand + (kThreads / 32) - 1) / (kThreads / 32);
    const dim3 g(static_cast<unsigned>(blocks_needed < static_cast<int64_t>(sms) * 8 ? blocks_needed : static_cast<int64_t>(sms) * 8));
    const bool cosine = metric == FFR_METRIC_COSINE;
    // the self kernel reads its references from global memory, in the form of K2s's scan of more than two references (the
    // form the tcgen05 Euclid value pass reproduces), whatever n is
    const int mode = k2s_form(x, cand, INT64_MAX, dim);
#define FFR_SELF_LAUNCH(NV)                                                                                                   \
    if (cosine) filter_fp32_kernel<NV, true, 0, true><<<g, kThreads, 0, s>>>(x, n, cand, n_cand, dim, thr, 0, o.keep, o.idx, o.val, o.band, self);  \
    else        filter_fp32_kernel<NV, false, 0, true><<<g, kThreads, 0, s>>>(x, n, cand, n_cand, dim, thr, 0, o.keep, o.idx, o.val, o.band, self)
    switch (mode) {
        case 1: FFR_SELF_LAUNCH(1); break;
        case 2: FFR_SELF_LAUNCH(2); break;
        case 4: FFR_SELF_LAUNCH(4); break;
        case 8: FFR_SELF_LAUNCH(8); break;
        default:
            if (cosine) filter_fp32_generic_kernel<true, true><<<g, kThreads, 0, s>>>(x, n, cand, n_cand, dim, thr, 0, o.keep, o.idx, o.val, o.band, self);
            else        filter_fp32_generic_kernel<false, true><<<g, kThreads, 0, s>>>(x, n, cand, n_cand, dim, thr, 0, o.keep, o.idx, o.val, o.band, self);
    }
#undef FFR_SELF_LAUNCH
    FFR_LAUNCH_CHECK("filter_fp32_self");
    return FFR_OK;
}

int launch_ref_stats(const float* ref_feat, int32_t n_ref, int32_t dim, float* mean, float* thres, cudaStream_t s) {
    const size_t smem = (static_cast<size_t>(dim) + 8) * sizeof(float);
    ref_stats_kernel<<<1, 256, smem, s>>>(ref_feat, n_ref, dim, mean, thres, k2s_form(ref_feat, ref_feat, 1, dim));
    FFR_LAUNCH_CHECK("ref_stats");
    return FFR_OK;
}

}  // namespace ffr

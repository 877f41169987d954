// K1 -- row L2-normalisation of an embedding matrix, sm_100a.
//
// Replaces  face_detection_and_extraction/modules/mobile_facenet/mobile_facenet.py:30-33 (l2_norm:
// norm = torch.norm(x, 2, axis, True); x / norm) and
// face_detection_and_extraction/face_extraction/extract_and_clean_imdb_wiki_faces.py:146
// (face_feat / np.linalg.norm(face_feat)).  No epsilon, true IEEE division, like the reference.
//
// HBM-bound: reads 4*dim bytes per row, writes 2*ld16 (fp16 copy for the tensor-core filter) and/or
// 4*dim (fp32 copy) and 4 (norm).  One warp owns one row at a time: lane l loads float4 #(l + 32 j) of
// the row (fully coalesced 512 B per warp instruction, streaming / no L1 allocation), the sum of squares
// is reduced with warp shuffles, and each lane normalises and stores what it loaded.  Two rows are in
// flight per warp iteration to keep enough loads outstanding; the grid is a multiple of the SM count and
// warps stride over rows.
#include <stdlib.h>

#include "ffr_common.cuh"

namespace ffr {

namespace {

constexpr int kThreads = 256;           // 8 warps per CTA
constexpr int kRowsPerIter = 2;        // generic kernel / grid sizing; the vector kernel keeps >= 2 KB per warp in flight

// Optional second matrix (x_b, rows_b -> y16_b; fp16 output only): the filter normalises references and candidates in
// ONE launch -- virtual rows [0, rows) are matrix a, [rows, rows + rows_b) matrix b -- and the same launch zeroes the
// re-check header K2 appends to (zero_words 32-bit words at zero_ptr), saving a launch and a memset per call.
struct L2Second {
    const float* x;
    int64_t rows;
    __half* y16;
    uint32_t* zero_ptr;
    int32_t zero_words;
    float* scale_a;           // optional: 1 / |x| of matrix a's rows (the Euclid filter's candidate scales)
};

template <int NV, int kRows>             // NV float4 per lane per row (dim == 128 * NV), kRows rows in flight per warp
__global__ void __launch_bounds__(kThreads)
l2norm_rows_vec_kernel(const float* __restrict__ x_a, int64_t rows_a, int32_t dim,
                       __half* __restrict__ y16_a, int32_t ld16, float* __restrict__ y32,
                       float* __restrict__ norms, const L2Second sec) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;
    pdl_launch_dependents();            // K2 may start its prologue / candidate staging now; it waits (pdl_wait) before it reads our output
    if (blockIdx.x == 0 && threadIdx.x < sec.zero_words) sec.zero_ptr[threadIdx.x] = 0u;
    const int64_t rows = rows_a + sec.rows;

    for (int64_t r0 = warp * kRows; r0 < rows; r0 += nwarps * kRows) {
        float4 v[kRows][NV];
#pragma unroll
        for (int i = 0; i < kRows; ++i) {
            const int64_t r = r0 + i;
            if (r < rows) {
                const float4* p = reinterpret_cast<const float4*>(r < rows_a ? x_a + r * dim : sec.x + (r - rows_a) * dim);
#pragma unroll
                for (int j = 0; j < NV; ++j) v[i][j] = ldg_stream_f4(p + lane + 32 * j);
            }
        }
#pragma unroll
        for (int i = 0; i < kRows; ++i) {
            const int64_t r = r0 + i;
            if (r >= rows) break;
            float ss = 0.f;
#pragma unroll
            for (int j = 0; j < NV; ++j) {
                ss = fmaf(v[i][j].x, v[i][j].x, ss);
                ss = fmaf(v[i][j].y, v[i][j].y, ss);
                ss = fmaf(v[i][j].z, v[i][j].z, ss);
                ss = fmaf(v[i][j].w, v[i][j].w, ss);
            }
            ss = warp_sum(ss);
            const float nrm = sqrtf(ss);
            if (norms != nullptr && lane == 0) norms[r] = nrm;
            if (sec.scale_a != nullptr && lane == 0 && r < rows_a) sec.scale_a[r] = __fdiv_rn(1.0f, nrm);
            __half* y16 = y16_a;
            int64_t ro = r;                                         // row inside its own matrix
            if (r >= rows_a) { y16 = sec.y16; ro = r - rows_a; }
#pragma unroll
            for (int j = 0; j < NV; ++j) {
                float4 o;
                o.x = __fdiv_rn(v[i][j].x, nrm);
                o.y = __fdiv_rn(v[i][j].y, nrm);
                o.z = __fdiv_rn(v[i][j].z, nrm);
                o.w = __fdiv_rn(v[i][j].w, nrm);
                if (y32 != nullptr) reinterpret_cast<float4*>(y32 + r * dim)[lane + 32 * j] = o;
                if (y16 != nullptr) {
                    __half2 h0 = __floats2half2_rn(o.x, o.y);
                    __half2 h1 = __floats2half2_rn(o.z, o.w);
                    uint2 pk;
                    pk.x = *reinterpret_cast<uint32_t*>(&h0);
                    pk.y = *reinterpret_cast<uint32_t*>(&h1);
                    reinterpret_cast<uint2*>(y16 + ro * ld16)[lane + 32 * j] = pk;
                }
            }
            if (y16 != nullptr) {                                   // zero the K padding (dim..ld16)
                for (int c = dim + lane * 4; c < ld16; c += 128)
                    *reinterpret_cast<uint2*>(y16 + ro * ld16 + c) = make_uint2(0u, 0u);
            }
        }
    }
}

// Short rows (dim 128 / 256), fp16 output only: a row is owned by L = dim / 16 lanes (4 float4 each), so a warp
// instruction covers 32 / L rows and the sum of squares needs log2(L) shuffles.  The warp-per-row kernel above spends
// ~70 instructions per 128-d row (five shuffles, a sqrt and four IEEE divisions per lane for ONE float4) and is issue
// bound at 3.2 TB/s; here a row costs ~15.  One IEEE reciprocal per row, then multiplies (<= 1.5 ulp from x / |x| before
// the fp16 rounding -- the same arithmetic as K2's normaliser warps).
template <int L>
__global__ void __launch_bounds__(kThreads)
l2norm_rows_sub_kernel(const float* __restrict__ x_a, int64_t rows_a, int32_t dim, __half* __restrict__ y16_a, int32_t ld16,
                       const L2Second sec) {
    constexpr int kRowsPerWarp = 32 / L;
    constexpr int kGroups = 2;                                      // row groups in flight per warp (4 KB)
    const int lane = threadIdx.x & 31, sub = lane % L, rsel = lane / L;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;
    pdl_launch_dependents();            // K2 may start its prologue / candidate staging now; it waits (pdl_wait) before it reads our output
    if (blockIdx.x == 0 && threadIdx.x < sec.zero_words) sec.zero_ptr[threadIdx.x] = 0u;
    const int64_t rows = rows_a + sec.rows;
    for (int64_t r0 = warp * (kGroups * kRowsPerWarp); r0 < rows; r0 += nwarps * (kGroups * kRowsPerWarp)) {
        float4 v[kGroups][4];
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const int64_t r = r0 + g * kRowsPerWarp + rsel;
            if (r < rows) {
                const float4* p = reinterpret_cast<const float4*>(r < rows_a ? x_a + r * dim : sec.x + (r - rows_a) * dim);
#pragma unroll
                for (int j = 0; j < 4; ++j) v[g][j] = ldg_stream_f4(p + sub + L * j);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) v[g][j] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const int64_t r = r0 + g * kRowsPerWarp + rsel;
            float ss = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                ss = fmaf(v[g][j].x, v[g][j].x, ss); ss = fmaf(v[g][j].y, v[g][j].y, ss);
                ss = fmaf(v[g][j].z, v[g][j].z, ss); ss = fmaf(v[g][j].w, v[g][j].w, ss);
            }
#pragma unroll
            for (int o = L / 2; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
            const float inv = __fdiv_rn(1.0f, sqrtf(ss));
            if (sec.scale_a != nullptr && sub == 0 && r < rows_a) sec.scale_a[r] = inv;
            if (r < rows) {
                __half* y = (r < rows_a) ? y16_a + r * ld16 : sec.y16 + (r - rows_a) * ld16;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const __half2 h0 = __floats2half2_rn(v[g][j].x * inv, v[g][j].y * inv);
                    const __half2 h1 = __floats2half2_rn(v[g][j].z * inv, v[g][j].w * inv);
                    uint2 pk;
                    pk.x = *reinterpret_cast<const uint32_t*>(&h0);
                    pk.y = *reinterpret_cast<const uint32_t*>(&h1);
                    reinterpret_cast<uint2*>(y)[sub + L * j] = pk;
                }
            }
        }
    }
}

// any dim: one warp per row, scalar accesses (row may be unaligned for float4)
__global__ void __launch_bounds__(kThreads)
l2norm_rows_generic_kernel(const float* __restrict__ x_a, int64_t rows_a, int32_t dim,
                           __half* __restrict__ y16_a, int32_t ld16, float* __restrict__ y32,
                           float* __restrict__ norms, const L2Second sec) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;
    pdl_launch_dependents();            // K2 may start its prologue / candidate staging now; it waits (pdl_wait) before it reads our output
    if (blockIdx.x == 0 && threadIdx.x < sec.zero_words) sec.zero_ptr[threadIdx.x] = 0u;
    const int64_t rows = rows_a + sec.rows;
    for (int64_t rv = warp; rv < rows; rv += nwarps) {
        const bool second = rv >= rows_a;
        const int64_t r = second ? rv - rows_a : rv;
        const float* p = second ? sec.x + r * dim : x_a + r * dim;
        __half* y16 = second ? sec.y16 : y16_a;
        float ss = 0.f;
        for (int c = lane; c < dim; c += 32) { const float t = __ldg(p + c); ss = fmaf(t, t, ss); }
        ss = warp_sum(ss);
        const float nrm = sqrtf(ss);
        if (norms != nullptr && lane == 0) norms[r] = nrm;
        if (sec.scale_a != nullptr && lane == 0 && !second) sec.scale_a[r] = __fdiv_rn(1.0f, nrm);
        for (int c = lane; c < ld16 || c < dim; c += 32) {
            const float o = c < dim ? __fdiv_rn(__ldg(p + c), nrm) : 0.f;
            if (y32 != nullptr && c < dim) y32[r * dim + c] = o;
            if (y16 != nullptr && c < ld16) y16[r * ld16 + c] = __float2half_rn(o);
        }
    }
}

static int launch_l2norm_impl(const float* x, int64_t rows, int32_t dim, __half* y16, int32_t ld16, float* y32, float* norms,
                              const L2Second sec, cudaStream_t s) {
    if (rows + sec.rows == 0 && sec.zero_words == 0) return FFR_OK;
    const int sms = num_sms();
    const int64_t warps_needed = (rows + sec.rows + kRowsPerIter - 1) / kRowsPerIter;
    const int64_t blocks_needed = (warps_needed + (kThreads / 32) - 1) / (kThreads / 32);
    // up to 8 resident CTAs per SM (2048 threads); whole multiples of the SM count when the matrix is big
    int64_t grid = blocks_needed < static_cast<int64_t>(sms) * 8 ? blocks_needed : static_cast<int64_t>(sms) * 8;
    if (grid < 1) grid = 1;
    const bool vec_ok = (dim % 128 == 0) && (y16 == nullptr || (ld16 % 4 == 0)) &&
                        ((reinterpret_cast<uintptr_t>(x) & 15) == 0) &&
                        (y32 == nullptr || (reinterpret_cast<uintptr_t>(y32) & 15) == 0) &&
                        (y16 == nullptr || (reinterpret_cast<uintptr_t>(y16) & 7) == 0) &&
                        (sec.rows == 0 || ((reinterpret_cast<uintptr_t>(sec.x) & 15) == 0 &&
                                           (reinterpret_cast<uintptr_t>(sec.y16) & 7) == 0));
    const dim3 g(static_cast<unsigned>(grid)), b(kThreads);
    const bool sub_ok = vec_ok && y32 == nullptr && norms == nullptr && y16 != nullptr && ld16 == dim;
    if (sub_ok && (dim == 128 || dim == 256)) {
        // 8 rows (dim 128) / 4 rows (dim 256) per warp iteration
        const int64_t rows_per_warp = (dim == 128 ? 4 : 2) * 2;
        const int64_t w_needed = (rows + sec.rows + rows_per_warp - 1) / rows_per_warp;
        int64_t gsub = (w_needed + (kThreads / 32) - 1) / (kThreads / 32);
        if (gsub > static_cast<int64_t>(sms) * 8) gsub = static_cast<int64_t>(sms) * 8;
        if (gsub < 1) gsub = 1;
        const dim3 gs(static_cast<unsigned>(gsub));
        if (dim == 128) l2norm_rows_sub_kernel<8><<<gs, b, 0, s>>>(x, rows, dim, y16, ld16, sec);
        else            l2norm_rows_sub_kernel<16><<<gs, b, 0, s>>>(x, rows, dim, y16, ld16, sec);
        FFR_LAUNCH_CHECK("l2norm_rows_sub");
        return FFR_OK;
    }
    if (vec_ok && dim == 128)       l2norm_rows_vec_kernel<1, 8><<<g, b, 0, s>>>(x, rows, dim, y16, ld16, y32, norms, sec);
    else if (vec_ok && dim == 256)  l2norm_rows_vec_kernel<2, 4><<<g, b, 0, s>>>(x, rows, dim, y16, ld16, y32, norms, sec);
    else if (vec_ok && dim == 384)  l2norm_rows_vec_kernel<3, 2><<<g, b, 0, s>>>(x, rows, dim, y16, ld16, y32, norms, sec);
    else if (vec_ok && dim == 512)  l2norm_rows_vec_kernel<4, 2><<<g, b, 0, s>>>(x, rows, dim, y16, ld16, y32, norms, sec);
    else if (vec_ok && dim == 1024) l2norm_rows_vec_kernel<8, 1><<<g, b, 0, s>>>(x, rows, dim, y16, ld16, y32, norms, sec);
    else l2norm_rows_generic_kernel<<<g, b, 0, s>>>(x, rows, dim, y16, ld16, y32, norms, sec);
    FFR_LAUNCH_CHECK("l2norm_rows");
    return FFR_OK;
}

}  // namespace

int launch_l2norm(const float* x, int64_t rows, int32_t dim, __half* y16, int32_t ld16, float* y32, float* norms,
                  cudaStream_t s) {
    return launch_l2norm_impl(x, rows, dim, y16, ld16, y32, norms, L2Second{nullptr, 0, nullptr, nullptr, 0, nullptr}, s);
}

// fp16 normalised copies of two matrices of the same width in one launch (either may be empty), plus zero_words 32-bit
// zeros at zero_ptr (<= 256 words)
int launch_l2norm_pair(const float* x_a, int64_t rows_a, __half* y16_a, const float* x_b, int64_t rows_b, __half* y16_b,
                       int32_t dim, int32_t ld16, void* zero_ptr, int32_t zero_words, cudaStream_t s, float* scale_a) {
    return launch_l2norm_impl(x_a, rows_a, dim, y16_a, ld16, nullptr, nullptr,
                              L2Second{x_b, rows_b, y16_b, static_cast<uint32_t*>(zero_ptr), zero_words, scale_a}, s);
}

// ---- Euclid references for the tensor-core filter (DESIGN.md section 4, "Euclid on the tensor cores") ----
// argmin_i |c - r_i| = argmax_i (r_i.c - |r_i|^2 / 2).  K2 multiplies fp16(r * 2^-f) by the candidate's normalised fp16 row
// and adds beta_i / |c|, beta_i = -|r_i|^2 * 2^-f / 2.  One power of two f per call, from the largest reference norm, keeps
// |r * 2^-f| <= 1, so the fp16 operand error is bounded like the cosine score's.  The squares are summed in fp64 and rounded
// once: beta then carries a single fp32 rounding, which is what K2's per-row window accounts for.
// E1: one warp per row, |r_i|^2 and the running maximum (the bits of non-negative floats order like the floats).
__global__ void __launch_bounds__(kThreads)
euclid_ref_norms_kernel(const float* __restrict__ ref, int64_t n_ref, int32_t dim, float* __restrict__ nsq,
                        uint32_t* __restrict__ max_bits) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;
    for (int64_t r = warp; r < n_ref; r += nwarps) {
        const float* p = ref + r * dim;
        double ss = 0.0;
        for (int c = lane; c < dim; c += 32) { const double t = __ldg(p + c); ss = fma(t, t, ss); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if (lane == 0) {
            const float v = static_cast<float>(ss);
            nsq[r] = v;
            atomicMax(max_bits, __float_as_uint(v));
        }
    }
}

// E2: f = the smallest integer with 2^(2f) > max |r|^2; fp16(r * 2^-f) rows (zero K padding), beta (zero padded to a multiple
// of 256 so that K2's reads of a partial reference tile stay inside the tensor), bmax = max |beta|.
__global__ void __launch_bounds__(kThreads)
euclid_ref_scale_kernel(const float* __restrict__ ref, int64_t n_ref, int32_t dim, int32_t ld16, __half* __restrict__ ref16,
                        const float* __restrict__ nsq, const uint32_t* __restrict__ max_bits, float* __restrict__ beta,
                        int64_t n_pad, float* __restrict__ bmax) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;
    const float mx = __uint_as_float(*max_bits);
    const float sc = euclid_ref_scale(mx);
    if (blockIdx.x == 0 && threadIdx.x == 0) *bmax = 0.5f * (mx * sc);
    for (int64_t r = warp; r < n_pad; r += nwarps) {
        if (r >= n_ref) { if (lane == 0) beta[r] = 0.f; continue; }
        const float* p = ref + r * dim;
        __half* y = ref16 + r * ld16;
        for (int c = lane; c < ld16; c += 32) y[c] = __float2half_rn(c < dim ? __ldg(p + c) * sc : 0.f);
        if (lane == 0) beta[r] = -0.5f * (nsq[r] * sc);
    }
}

int launch_euclid_refs(const float* ref, int64_t n_ref, int32_t dim, int32_t ld16, __half* ref16, float* beta, float* nsq,
                       uint32_t* max_bits, float* bmax, cudaStream_t s) {
    const int64_t n_pad = euclid_bias_len(n_ref);
    int64_t grid = (n_pad + (kThreads / 32) - 1) / (kThreads / 32);
    if (grid > static_cast<int64_t>(num_sms()) * 8) grid = static_cast<int64_t>(num_sms()) * 8;
    FFR_CUDA_TRY(cudaMemsetAsync(max_bits, 0, sizeof(uint32_t), s));
    euclid_ref_norms_kernel<<<static_cast<unsigned>(grid), kThreads, 0, s>>>(ref, n_ref, dim, nsq, max_bits);
    FFR_LAUNCH_CHECK("euclid_ref_norms");
    euclid_ref_scale_kernel<<<static_cast<unsigned>(grid), kThreads, 0, s>>>(ref, n_ref, dim, ld16, ref16, nsq, max_bits, beta,
                                                                             n_pad, bmax);
    FFR_LAUNCH_CHECK("euclid_ref_scale");
    return FFR_OK;
}

}  // namespace ffr

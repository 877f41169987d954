// Exact-duplicate reference rows are folded before the tensor-core scan (round 2: the "K3 cliff").
//
// A gallery that holds the same embedding several times (the same photo enrolled again: the realistic case for face data)
// gives every candidate of that identity several EXACTLY equal leading scores.  K2 tracks three candidates per row; a
// fourth one inside the window sends the row to K3's fp32 rescan of the whole reference set, and with enough such rows K3
// costs many times K2.  np.argmax's first-occurrence rule -- the rule the best-match index follows (oracle.filter_cosine;
// the scan replaced is extract_and_label_faces_from_dataset.py:101-116) -- means a later bit-identical copy of a row can
// never be the answer: it is dropped here, K2 scans the unique rows only (fewer MMAs, no artificial ties) and maps its
// column indices back through `map`.  Order is preserved, so "ascending index = first occurrence" still holds.
//
//   D1 hash_rows_kernel     one warp per row: 64-bit hash of the row's bits, open-addressing insert keyed by the hash,
//                           value = smallest row index with that hash (atomicMin)
//   D2 mark_dups_kernel     one warp per row: the representative of its hash; bit-for-bit comparison of the two rows
//                           (a hash collision between different rows keeps both: dedup is an optimisation, never a guess)
//   D3 scan_unique_kernel   exclusive prefix sum of the "unique" flags (one CTA), number of unique rows
//   D4 compact_rows_kernel  unique fp16 rows (K1's output) -> consecutive rows; map[new] = old; with the Euclid filter the
//                           per-reference bias moves with its row
#include "ffr_common.cuh"

namespace ffr {

namespace {

constexpr int kThreads = 256;
constexpr unsigned long long kMul = 0x9E3779B97F4A7C15ull;

__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
    x ^= x >> 32; x *= 0xD6E8FEB86659FD93ull;
    x ^= x >> 32; x *= 0xD6E8FEB86659FD93ull;
    x ^= x >> 32;
    return x;
}

__global__ void __launch_bounds__(kThreads)
hash_rows_kernel(const float* __restrict__ x, int64_t rows, int32_t dim, unsigned long long* __restrict__ hashes,
                 unsigned long long* __restrict__ keys, int32_t* __restrict__ vals, uint32_t mask) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;
    for (int64_t r = warp; r < rows; r += nwarps) {
        const uint32_t* p = reinterpret_cast<const uint32_t*>(x + r * dim);
        unsigned long long h = 0x243F6A8885A308D3ull + static_cast<unsigned long long>(lane);
        for (int k = lane; k < dim; k += 32) h = (h ^ __ldg(p + k)) * kMul + static_cast<unsigned long long>(k);
        h = mix64(h);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
        h = mix64(h) | (1ull << 63);                                  // never 0 (0 = empty slot)
        if (lane == 0) {
            hashes[r] = h;
            uint32_t slot = static_cast<uint32_t>(h) & mask;
            while (true) {
                const unsigned long long prev = atomicCAS(&keys[slot], 0ull, h);
                if (prev == 0ull || prev == h) { atomicMin(&vals[slot], static_cast<int32_t>(r)); break; }
                slot = (slot + 1) & mask;
            }
        }
    }
}

__global__ void __launch_bounds__(kThreads)
mark_dups_kernel(const float* __restrict__ x, int64_t rows, int32_t dim, const unsigned long long* __restrict__ hashes,
                 const unsigned long long* __restrict__ keys, const int32_t* __restrict__ vals, uint32_t mask,
                 int32_t* __restrict__ unique) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;
    for (int64_t r = warp; r < rows; r += nwarps) {
        const unsigned long long h = hashes[r];
        uint32_t slot = static_cast<uint32_t>(h) & mask;
        while (keys[slot] != h) slot = (slot + 1) & mask;              // present: D1 inserted it
        const int64_t rep = vals[slot];
        bool same = rep < r;
        if (same) {
            const uint32_t* a = reinterpret_cast<const uint32_t*>(x + r * dim);
            const uint32_t* b = reinterpret_cast<const uint32_t*>(x + rep * dim);
            for (int k = lane; k < dim; k += 32) same = same && (__ldg(a + k) == __ldg(b + k));
        }
        same = __all_sync(0xffffffffu, same);
        if (lane == 0) unique[r] = same ? 0 : 1;
    }
}

// exclusive prefix sum of unique[0..rows) in place (unique[r] -> position of row r among the unique rows, or -1 for a
// duplicate), *n_unique = number of unique rows.  One CTA of 32 warps: every warp owns a contiguous segment and walks it 32
// elements at a time (coalesced loads, warp-shuffle scan, running carry) -- once to sum it, once to write the positions.
// (The first version gave every THREAD a contiguous run: 94 us for 100 k references, all of it uncoalesced latency.)
__global__ void __launch_bounds__(1024)
scan_unique_kernel(int32_t* __restrict__ unique, int64_t rows, int32_t* __restrict__ n_unique) {
    __shared__ int32_t s_part[32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t per = ((rows + 31) / 32 + 31) / 32 * 32;                  // segment length per warp, a multiple of 32
    const int64_t lo = w * per, hi = lo + per < rows ? lo + per : rows;
    int32_t sum = 0;
    for (int64_t i = lo + lane; i < hi; i += 32) sum += unique[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) s_part[w] = sum;
    __syncthreads();
    if (w == 0) {                                                           // exclusive scan of the 32 segment sums
        const int32_t v = s_part[lane];
        int32_t inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int32_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        s_part[lane] = inc - v;
        if (lane == 31) *n_unique = inc;
    }
    __syncthreads();
    int32_t carry = s_part[w];
    for (int64_t i0 = lo; i0 < hi; i0 += 32) {
        const int64_t i = i0 + lane;
        const int32_t u = i < hi ? unique[i] : 0;
        int32_t inc = u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int32_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (i < hi) unique[i] = u ? carry + inc - u : -1;
        carry += __shfl_sync(0xffffffffu, inc, 31);
    }
}

__global__ void __launch_bounds__(kThreads)
compact_rows_kernel(const __half* __restrict__ src, int64_t rows, int32_t ld, const int32_t* __restrict__ pos,
                    __half* __restrict__ dst, int32_t* __restrict__ map, const float* __restrict__ bias,
                    float* __restrict__ bias_c) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * kThreads) >> 5;
    const int n16 = ld / 8;                                             // ld is a multiple of 64 halves: 16-byte pieces
    for (int64_t r = warp; r < rows; r += nwarps) {
        const int32_t q = pos[r];
        if (q < 0) continue;
        const uint4* s = reinterpret_cast<const uint4*>(src + r * ld);
        uint4* d = reinterpret_cast<uint4*>(dst + static_cast<int64_t>(q) * ld);
        for (int k = lane; k < n16; k += 32) d[k] = __ldg(s + k);
        if (lane == 0) map[q] = static_cast<int32_t>(r);
        if (lane == 0 && bias != nullptr) bias_c[q] = bias[r];
    }
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

uint32_t table_size(int64_t n_ref) {
    uint32_t t = 1024;
    while (t < 2 * static_cast<uint64_t>(n_ref)) t <<= 1;
    return t;
}

}  // namespace

bool dedup_wanted(int64_t n_ref, int64_t n_cand) {
    // four small launches + two memsets: only where K2 runs for a good fraction of a millisecond anyway
    return knobs().dedup_refs != 0 && n_ref >= 2048 && n_ref < (int64_t(1) << 30) &&
           static_cast<double>(n_ref) * static_cast<double>(n_cand) >= 2e9;
}

size_t dedup_workspace_bytes(int64_t n_ref, int32_t ld) {
    const size_t n = static_cast<size_t>(n_ref), t = table_size(n_ref);
    return align_up(n * 8, 256) + align_up(t * 8, 256) + align_up(t * 4, 256) + align_up((n + 1) * 4, 256) + align_up(n * 4, 256) +
           align_up(n * static_cast<size_t>(ld) * 2, 256);
}

// ref32: the original rows; ref16_full: K1's normalised fp16 rows of ALL references (leading dimension ld).  On return (stream
// order) *out_ref16 holds the unique rows, *out_map the compact -> original index map, *out_n_unique (device) their count.
int launch_dedup_refs(const float* ref32, const __half* ref16_full, int64_t n_ref, int32_t dim, int32_t ld, void* ws,
                      __half** out_ref16, int32_t** out_map, int32_t** out_n_unique_dev, cudaStream_t s,
                      const float* bias, float* bias_c) {
    uint8_t* w = static_cast<uint8_t*>(ws);
    const size_t n = static_cast<size_t>(n_ref);
    const uint32_t t = table_size(n_ref);
    unsigned long long* hashes = reinterpret_cast<unsigned long long*>(w); w += align_up(n * 8, 256);
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(w);   w += align_up(static_cast<size_t>(t) * 8, 256);
    int32_t* vals = reinterpret_cast<int32_t*>(w);                         w += align_up(static_cast<size_t>(t) * 4, 256);
    int32_t* pos = reinterpret_cast<int32_t*>(w);                          w += align_up((n + 1) * 4, 256);   // [n] positions, [n] = count
    int32_t* map = reinterpret_cast<int32_t*>(w);                          w += align_up(n * 4, 256);
    __half* ref16c = reinterpret_cast<__half*>(w);
    FFR_CUDA_TRY(cudaMemsetAsync(keys, 0, static_cast<size_t>(t) * 8, s));
    FFR_CUDA_TRY(cudaMemsetAsync(vals, 0x7f, static_cast<size_t>(t) * 4, s));
    const int sms = num_sms();
    int64_t grid = (n_ref + (kThreads / 32) - 1) / (kThreads / 32);
    if (grid > static_cast<int64_t>(sms) * 8) grid = static_cast<int64_t>(sms) * 8;
    const dim3 g(static_cast<unsigned>(grid));
    hash_rows_kernel<<<g, kThreads, 0, s>>>(ref32, n_ref, dim, hashes, keys, vals, t - 1);
    FFR_LAUNCH_CHECK("dedup_hash_rows");
    mark_dups_kernel<<<g, kThreads, 0, s>>>(ref32, n_ref, dim, hashes, keys, vals, t - 1, pos);
    FFR_LAUNCH_CHECK("dedup_mark_dups");
    scan_unique_kernel<<<1, 1024, 0, s>>>(pos, n_ref, pos + n_ref);
    FFR_LAUNCH_CHECK("dedup_scan_unique");
    compact_rows_kernel<<<g, kThreads, 0, s>>>(ref16_full, n_ref, ld, pos, ref16c, map, bias, bias_c);
    FFR_LAUNCH_CHECK("dedup_compact_rows");
    *out_ref16 = ref16c;
    *out_map = map;
    *out_n_unique_dev = pos + n_ref;
    return FFR_OK;
}

}  // namespace ffr

// K3 -- fp32 re-check of the rows K2 flagged, and K4's pack/unpack helpers.
//
// K2 scores with fp16-rounded operands.  The parity contract (BASELINE.md) wants keep masks and best-match
// indices equal to the reference's fp32 cosine path (extract_and_label_faces_from_dataset.py:106 evaluated
// in fp32), so every row whose decision could be changed by the rounding -- top-2 gap <= delta, or best
// within the band of the threshold -- is recomputed here with the reference's own formula
//     inner(f, g) / (|f| * |g|)
// on the ORIGINAL fp32 embeddings: only the two leading references when the third-best score was clearly
// lower, the whole reference set otherwise (first-occurrence argmax, strict '>' in ascending order).
// One warp per flagged row; the candidate row is parked in shared memory.
//
// Euclid form (kEuclid, the tcgen05 Euclid filter): the same lists, ranked by fp32 distance computed with direct differences
// (c - r, never |c|^2 + |r|^2 - 2 c.r), smallest first, ties to the first index.  Only best_idx is written: keep, best_val and
// the band come from the value pass that follows (ffr_filter_fp32.cu), which recomputes the winner's distance with K2s's
// arithmetic.  The pairs, parts and few-row phases use k2s_euclid_dist in K2s's mode (`emode`); the tiled walk has its own
// difference-and-square loop.
#include <mutex>

#include "ffr_common.cuh"

namespace ffr {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kKC = 8;             // floats per staged reference chunk (two float4)
constexpr int kKCPad = 12;         // padded row stride (48 B): conflict-free float4 reads, 16-byte aligned
constexpr int kRefsPerThread = 2;  // register tile: 2 references x kFullGroup (16) candidates per thread
constexpr int kTileRefs = kThreads * kRefsPerThread;   // 1024 references staged per tile

__device__ __forceinline__ float cos_fp32(const float* __restrict__ c_smem, const float* __restrict__ r, int32_t dim,
                                          float cc_sqrt, int lane, bool vec) {
    float a = 0.f, b = 0.f;
    if (vec) {
        const float4* r4 = reinterpret_cast<const float4*>(r);
        const float4* c4 = reinterpret_cast<const float4*>(c_smem);
        for (int k = lane; k < (dim >> 2); k += 32) {
            const float4 rv = __ldg(r4 + k);
            const float4 cv = c4[k];
            a = fmaf(cv.x, rv.x, a); a = fmaf(cv.y, rv.y, a); a = fmaf(cv.z, rv.z, a); a = fmaf(cv.w, rv.w, a);
            b = fmaf(rv.x, rv.x, b); b = fmaf(rv.y, rv.y, b); b = fmaf(rv.z, rv.z, b); b = fmaf(rv.w, rv.w, b);
        }
    } else {
        for (int k = lane; k < dim; k += 32) {
            const float rv = __ldg(r + k), cv = c_smem[k];
            a = fmaf(cv, rv, a);
            b = fmaf(rv, rv, b);
        }
    }
    a = warp_sum(a);
    b = warp_sum(b);
    return __fdiv_rn(a, __fmul_rn(__fsqrt_rn(b), cc_sqrt));
}

// R consecutive reference rows at once (first row r0, row pitch dim; rows >= n_rows are clamped and their result is
// unused): the R loads per step are independent and the 2R shuffle reductions interleave, so a warp pays one memory
// latency and one reduction latency per R references instead of per reference -- the serial form made the few-row
// rescan pure latency (~1000 cycles per reference).  Same arithmetic per reference as cos_fp32.
template <int R>
__device__ __forceinline__ void cos_fp32_ptrs(const float* __restrict__ c_smem, const float* const (&rp)[R], int32_t dim,
                                              float cc_sqrt, int lane, bool vec, float (&out)[R]) {
    float a[R], b[R];
#pragma unroll
    for (int r = 0; r < R; ++r) { a[r] = 0.f; b[r] = 0.f; }
    if (vec) {
        const float4* c4 = reinterpret_cast<const float4*>(c_smem);
        for (int k = lane; k < (dim >> 2); k += 32) {
            const float4 cv = c4[k];
            float4 rv[R];
#pragma unroll
            for (int r = 0; r < R; ++r) rv[r] = __ldg(reinterpret_cast<const float4*>(rp[r]) + k);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                a[r] = fmaf(cv.x, rv[r].x, a[r]); a[r] = fmaf(cv.y, rv[r].y, a[r]);
                a[r] = fmaf(cv.z, rv[r].z, a[r]); a[r] = fmaf(cv.w, rv[r].w, a[r]);
                b[r] = fmaf(rv[r].x, rv[r].x, b[r]); b[r] = fmaf(rv[r].y, rv[r].y, b[r]);
                b[r] = fmaf(rv[r].z, rv[r].z, b[r]); b[r] = fmaf(rv[r].w, rv[r].w, b[r]);
            }
        }
    } else {
        for (int k = lane; k < dim; k += 32) {
            const float cv = c_smem[k];
            float rv[R];
#pragma unroll
            for (int r = 0; r < R; ++r) rv[r] = __ldg(rp[r] + k);
#pragma unroll
            for (int r = 0; r < R; ++r) { a[r] = fmaf(cv, rv[r], a[r]); b[r] = fmaf(rv[r], rv[r], b[r]); }
        }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) { a[r] = warp_sum(a[r]); b[r] = warp_sum(b[r]); }
#pragma unroll
    for (int r = 0; r < R; ++r) out[r] = __fdiv_rn(a[r], __fmul_rn(__fsqrt_rn(b[r]), cc_sqrt));
}

template <int R>
__device__ __forceinline__ void cos_fp32_multi(const float* __restrict__ c_smem, const float* __restrict__ r0, int n_rows,
                                               int32_t dim, float cc_sqrt, int lane, bool vec, float (&out)[R]) {
    const float* rp[R];
#pragma unroll
    for (int r = 0; r < R; ++r) rp[r] = r0 + static_cast<int64_t>(r < n_rows ? r : n_rows - 1) * dim;
    cos_fp32_ptrs<R>(c_smem, rp, dim, cc_sqrt, lane, vec, out);
}

__device__ __forceinline__ void emit_result(int32_t row, float best, int32_t bi, float thr, int64_t ref_index_base,
                                            uint8_t* keep, int32_t* best_idx, float* best_val, float band_tol,
                                            int32_t* band_count, int64_t* band_rows, int64_t band_cap) {
    keep[row] = (best >= thr) ? 1 : 0;
    best_idx[row] = static_cast<int32_t>(bi + ref_index_base);
    if (best_val != nullptr) best_val[row] = best;
    if (band_count != nullptr && fabsf(best - thr) <= band_tol) {
        const int32_t slot = atomicAdd(band_count, 1);
        if (band_rows != nullptr && slot < band_cap) band_rows[slot] = row;
    }
}

// K3a: near-tie / near-threshold rows -- fp32 cosine against the one to three leading references. One warp per row.
__device__ __forceinline__ void
recheck_pairs_phase(float* s_rows, const float* __restrict__ ref, const float* __restrict__ cand, int32_t dim, float thr,
                    int64_t ref_index_base, uint8_t* __restrict__ keep, int32_t* __restrict__ best_idx,
                    float* __restrict__ best_val, const RecheckLists& lists, float band_tol, int32_t* band_count,
                    int64_t* band_rows, int64_t band_cap, bool vec, int emode) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    float* c_smem = s_rows + static_cast<size_t>(w) * dim;
    const int64_t warp = static_cast<int64_t>(blockIdx.x) * kWarps + w;
    const int64_t nwarps = static_cast<int64_t>(gridDim.x) * kWarps;
    if (emode >= 0) {                                           // Euclid: the one to three leading references by fp32 distance
        int64_t count = lists.hdr->recheck_count;
        if (count > lists.rec_cap) count = lists.rec_cap;
        for (int64_t k = warp; k < count; k += nwarps) {
            const RecheckRec rec = lists.recs[k];
            const float* c = cand + static_cast<int64_t>(rec.row) * dim;
            float best = k2s_euclid_dist(c, ref + static_cast<int64_t>(rec.idx1) * dim, dim, lane, emode);
            int32_t bi = rec.idx1;
            const int32_t more[2] = {rec.idx2, rec.idx2 >= 0 ? rec.idx3 : -1};
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                if (more[e] < 0) continue;
                const float d = k2s_euclid_dist(c, ref + static_cast<int64_t>(more[e]) * dim, dim, lane, emode);
                if (d < best || (d == best && more[e] < bi)) { best = d; bi = more[e]; }
            }
            if (lane == 0) best_idx[rec.row] = static_cast<int32_t>(bi + ref_index_base);
        }
        return;
    }
    // the warp's first record is requested TOGETHER with the list length, not after it (it is only used when it exists):
    // with a short list the phase is one chain of dependent memory latencies, and this takes one L2 round trip out of it
    RecheckRec rec0{};
    if (warp < lists.rec_cap) rec0 = lists.recs[warp];
    int64_t count = lists.hdr->recheck_count;
    if (count > lists.rec_cap) count = lists.rec_cap;
    // The candidate row of the NEXT record is fetched into registers (an HBM miss, ~1.5 us) while the current one is
    // scored, and the up-to-three references of a record are scored together (one L2 round trip): a warp's rows used to
    // cost three or four dependent memory latencies each.
    const bool pipe = vec && dim <= 512;
    const int nvec = dim >> 2;
    if (vec && nvec <= 32) {
        // Rows of <= 128 floats: ONE float4 per lane and row, everything in registers.  With a short list (BASELINE configs[1]:
        // one record per warp) the phase is a chain of dependent memory latencies, so it is made as short as it gets: the
        // candidate row (HBM) and the up-to-three reference rows (L2) are requested together.  Same arithmetic as cos_fp32 / the parked-row form below, bit for bit.
        int64_t k = warp;
        RecheckRec rec = rec0;
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4* cand4 = reinterpret_cast<const float4*>(cand);
        const float4* ref4 = reinterpret_cast<const float4*>(ref);
        while (k < count) {
            const bool live = lane < nvec;
            const int32_t i2 = rec.idx2 >= 0 ? rec.idx2 : rec.idx1;
            const int32_t i3 = rec.idx3 >= 0 ? rec.idx3 : i2;
            const float4 cv = live ? __ldg(cand4 + static_cast<int64_t>(rec.row) * nvec + lane) : z4;
            float4 rv[3];
            rv[0] = live ? __ldg(ref4 + static_cast<int64_t>(rec.idx1) * nvec + lane) : z4;
            rv[1] = live ? __ldg(ref4 + static_cast<int64_t>(i2) * nvec + lane) : z4;
            rv[2] = live ? __ldg(ref4 + static_cast<int64_t>(i3) * nvec + lane) : z4;
            const int64_t k_next = k + nwarps;
            RecheckRec rec_next = rec;
            if (k_next < count) rec_next = lists.recs[k_next];
            float cc = 0.f;
            cc = fmaf(cv.x, cv.x, cc); cc = fmaf(cv.y, cv.y, cc); cc = fmaf(cv.z, cv.z, cc); cc = fmaf(cv.w, cv.w, cc);
            float a[3], b[3];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                a[r] = 0.f; b[r] = 0.f;
                a[r] = fmaf(cv.x, rv[r].x, a[r]); a[r] = fmaf(cv.y, rv[r].y, a[r]);
                a[r] = fmaf(cv.z, rv[r].z, a[r]); a[r] = fmaf(cv.w, rv[r].w, a[r]);
                b[r] = fmaf(rv[r].x, rv[r].x, b[r]); b[r] = fmaf(rv[r].y, rv[r].y, b[r]);
                b[r] = fmaf(rv[r].z, rv[r].z, b[r]); b[r] = fmaf(rv[r].w, rv[r].w, b[r]);
            }
            const float cc_sqrt = __fsqrt_rn(warp_sum(cc));
#pragma unroll
            for (int r = 0; r < 3; ++r) { a[r] = warp_sum(a[r]); b[r] = warp_sum(b[r]); }
            float sc[3];
#pragma unroll
            for (int r = 0; r < 3; ++r) sc[r] = __fdiv_rn(a[r], __fmul_rn(__fsqrt_rn(b[r]), cc_sqrt));
            float best = sc[0];
            int32_t bi = rec.idx1;
            if (rec.idx2 >= 0) {
                if (sc[1] > best || (sc[1] == best && rec.idx2 < bi)) { best = sc[1]; bi = rec.idx2; }
                if (rec.idx3 >= 0 && (sc[2] > best || (sc[2] == best && rec.idx3 < bi))) { best = sc[2]; bi = rec.idx3; }
            }
            if (lane == 0)
                emit_result(rec.row, best, bi, thr, ref_index_base, keep, best_idx, best_val, band_tol, band_count,
                            band_rows, band_cap);
            k = k_next;
            rec = rec_next;
        }
        return;
    }
    float4 pre[4];
    RecheckRec rec{}, rec_next{};
    int64_t k = warp;
    auto prefetch = [&](const RecheckRec& r) {
        const float4* c4 = reinterpret_cast<const float4*>(cand + static_cast<int64_t>(r.row) * dim);
#pragma unroll
        for (int j = 0; j < 4; ++j) pre[j] = (lane + 32 * j < nvec) ? __ldg(c4 + lane + 32 * j) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    if (k < count) { rec = rec0; if (pipe) prefetch(rec); }
    while (k < count) {
        float cc = 0.f;
        __syncwarp();
        if (pipe) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (lane + 32 * j < nvec) reinterpret_cast<float4*>(c_smem)[lane + 32 * j] = pre[j];
                cc = fmaf(pre[j].x, pre[j].x, cc); cc = fmaf(pre[j].y, pre[j].y, cc);
                cc = fmaf(pre[j].z, pre[j].z, cc); cc = fmaf(pre[j].w, pre[j].w, cc);
            }
        } else {
            const float* c = cand + static_cast<int64_t>(rec.row) * dim;
            for (int d = lane; d < dim; d += 32) { const float t = __ldg(c + d); c_smem[d] = t; cc = fmaf(t, t, cc); }
        }
        __syncwarp();
        const int64_t k_next = k + nwarps;
        if (k_next < count) { rec_next = lists.recs[k_next]; if (pipe) prefetch(rec_next); }
        const float cc_sqrt = __fsqrt_rn(warp_sum(cc));
        float best;
        int32_t bi = rec.idx1;
        if (rec.idx2 < 0) {
            best = cos_fp32(c_smem, ref + static_cast<int64_t>(rec.idx1) * dim, dim, cc_sqrt, lane, vec);
        } else {
            const int32_t i3 = rec.idx3 >= 0 ? rec.idx3 : rec.idx2;
            const float* rp[3] = {ref + static_cast<int64_t>(rec.idx1) * dim, ref + static_cast<int64_t>(rec.idx2) * dim,
                                  ref + static_cast<int64_t>(i3) * dim};
            float sc[3];
            cos_fp32_ptrs<3>(c_smem, rp, dim, cc_sqrt, lane, vec, sc);
            best = sc[0];
            if (sc[1] > best || (sc[1] == best && rec.idx2 < bi)) { best = sc[1]; bi = rec.idx2; }
            if (rec.idx3 >= 0 && (sc[2] > best || (sc[2] == best && rec.idx3 < bi))) { best = sc[2]; bi = rec.idx3; }
        }
        if (lane == 0)
            emit_result(rec.row, best, bi, thr, ref_index_base, keep, best_idx, best_val, band_tol, band_count,
                        band_rows, band_cap);
        k = k_next;
        rec = rec_next;
    }
}

// K3b: rows with three or more references inside the window -- exact fp32 rescan of the WHOLE reference set.
// A block owns kFullGroup candidate rows (parked in shared memory) and one slice of the references; every thread
// walks its own reference rows (thread-per-reference: no shuffles, each reference row is read once per group and
// reused for all kFullGroup candidates), keeps a per-candidate best with strict '>' in ascending order, and the
// block/ slice results are merged with a 64-bit atomicMax on (orderable(score) << 32 | ~index), which implements
// "largest score, then smallest index" = np.argmax.  The last slice to arrive writes the outputs.
// The same key merges a gallery sharded over ranks (ffr_allreduce_best: one ncclMax over uint64, v = -distance for Euclid, key 0
// = no reference).  sharding.pack_best_keys is its Python twin for torch.distributed, with the top bit flipped so that a SIGNED
// int64 max orders the keys the same way.
__device__ __forceinline__ unsigned long long pack_key(float v, int32_t idx) {
    uint32_t u = __float_as_uint(v);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return (static_cast<unsigned long long>(u) << 32) | static_cast<unsigned long long>(0xFFFFFFFFu - static_cast<uint32_t>(idx));
}
__device__ __forceinline__ void unpack_key(unsigned long long k, float& v, int32_t& idx) {
    uint32_t u = static_cast<uint32_t>(k >> 32);
    u = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
    v = __uint_as_float(u);
    idx = static_cast<int32_t>(0xFFFFFFFFu - static_cast<uint32_t>(k & 0xFFFFFFFFull));
}

// K3p: rows whose un-inserted in-window columns all lie in ONE 128-reference part of K2's column grid (flag-only update path,
// DESIGN.md section 4) -- or in TWO ADJACENT parts (a group of near-identical references that straddles a part boundary: the two
// parts are seen by the two column halves of K2's epilogue and joined when their states are merged).  Record: idx1 = (first
// compact column of the first part >> 7) | Y-group mask << 24, idx3 = X-group mask, 16 bits per part (bit a: columns
// 8a..8a+7 of the 256-column span; Y bit b: column mod 8 == b) -- the in-window columns are among {8a + b} -- and idx2 = one
// tracked candidate outside the span.  fp32 cosine against exactly those references; first occurrence of the maximum.  One
// warp per record, L LANES PER REFERENCE (the candidate row broadcast from shared memory).  Typically 2-8 references.
__device__ __forceinline__ int64_t parts_first_item(int64_t warp, int64_t nwarps) { return nwarps - 1 - warp; }

// kSelf: the X / Y masks name a superset of the in-window columns, which can include the row's own column (and, in
// FFR_SELF_EARLIER, later ones): excluded references are skipped.
template <bool kSelf>
__device__ __forceinline__ void
recheck_parts_phase(float* s_rows, const float* __restrict__ ref, int64_t n_ref, const float* __restrict__ cand, int32_t dim,
                    float thr, int64_t ref_index_base, uint8_t* __restrict__ keep, int32_t* __restrict__ best_idx,
                    float* __restrict__ best_val, const RecheckLists& lists, float band_tol, int32_t* band_count,
                    int64_t* band_rows, int64_t band_cap, bool vec, const int32_t* __restrict__ ref_map,
                    const int32_t* __restrict__ n_unique_dev, int emode, SelfArgs self) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    float* c_smem = s_rows + static_cast<size_t>(w) * dim;
    // records are dealt from the LAST warp of the grid downwards: with a short pairs list (dealt from warp 0 upwards) the two
    // phases then run on different warps at the same time instead of one after the other on the same ones
    const int64_t nwarps = static_cast<int64_t>(gridDim.x) * kWarps;
    const int64_t warp = parts_first_item(static_cast<int64_t>(blockIdx.x) * kWarps + w, nwarps);
    RecheckRec rec0{};                                            // requested together with the count (see the pairs phase)
    if (warp < lists.rec_cap) rec0 = lists.recs[lists.rec_cap - 1 - warp];
    // duplicate references folded before K2: the part is a range of COMPACT columns (ref_map: column -> original reference)
    const int64_t n_cols = n_unique_dev != nullptr ? static_cast<int64_t>(__ldg(n_unique_dev)) : n_ref;
    int64_t count = lists.hdr->part_count;
    if (count > lists.rec_cap) count = lists.rec_cap;
    for (int64_t k = warp; k < count; k += nwarps) {
        const RecheckRec rec = k == warp ? rec0 : lists.recs[lists.rec_cap - 1 - k];
        const uint32_t xm = static_cast<uint32_t>(rec.idx3), ym = static_cast<uint32_t>(rec.idx1) >> 24;
        const int64_t col0 = static_cast<int64_t>(static_cast<uint32_t>(rec.idx1) & 0xFFFFFFu) << 7;   // first compact column of the (first) part
        const int ny = __popc(ym);
        const int n_in = __popc(xm) * ny;                         // candidate columns inside the part(s) (<= 256)
        const int n_all = n_in + (rec.idx2 >= 0 ? 1 : 0);         // + the tracked candidate outside it
        if (emode >= 0) {                                         // Euclid: one reference at a time, the whole warp on it
            const float* c = cand + static_cast<int64_t>(rec.row) * dim;
            float best = INFINITY;
            int32_t bi = 0x7FFFFFFF;
            for (int e = 0; e < n_all; ++e) {
                int64_t ri = -1;
                if (e < n_in) {
                    const int a = __fns(xm, 0, e / ny + 1), b = __fns(ym, 0, e % ny + 1);
                    const int64_t col = col0 + 8 * a + b;
                    if (col < n_cols) ri = ref_map != nullptr ? static_cast<int64_t>(__ldg(ref_map + col)) : col;
                } else {
                    ri = rec.idx2;
                }
                if constexpr (kSelf) ri = self_eligible(ri, self.row0 + rec.row, self.mode) ? ri : -1;
                if (ri < 0) continue;
                const float d = k2s_euclid_dist(c, ref + ri * dim, dim, lane, emode);
                if (d < best || (d == best && ri < bi)) { best = d; bi = static_cast<int32_t>(ri); }
            }
            if (lane == 0 && bi != 0x7FFFFFFF) best_idx[rec.row] = static_cast<int32_t>(bi + ref_index_base);
            continue;
        }
        unsigned long long key = 0ull;
        // L lanes per reference (the embedding split between them): with the typical 2-8 references of a record most lanes
        // would idle and every lane would walk a whole row -- four times the dependent L2 round trips
        const int L = n_all <= 8 ? 4 : (n_all <= 16 ? 2 : 1);
        const int per = 32 / L, sub = lane % L;
        // the reference this lane scores in batch eb of `per` references (-1: none)
        auto ref_of = [&](int eb) -> int64_t {
            const int e = eb * per + lane / L;
            if (e < n_in) {
                const int a = __fns(xm, 0, e / ny + 1), b = __fns(ym, 0, e % ny + 1);     // e-th (a, b) pair in ascending column order
                const int64_t col = col0 + 8 * a + b;
                if (col < n_cols) return ref_map != nullptr ? static_cast<int64_t>(__ldg(ref_map + col)) : col;
                return -1;
            }
            return (e == n_in && rec.idx2 >= 0) ? static_cast<int64_t>(rec.idx2) : -1;
        };
        const float* c = cand + static_cast<int64_t>(rec.row) * dim;
        float cc = 0.f;
        __syncwarp();
        for (int d = lane; d < dim; d += 32) { const float t = __ldg(c + d); c_smem[d] = t; cc = fmaf(t, t, cc); }
        __syncwarp();
        const float cc_sqrt = __fsqrt_rn(warp_sum(cc));
        for (int e0 = 0, eb = 0; e0 < n_all; e0 += per, ++eb) {   // `per` references at a time
            int64_t ri = ref_of(eb);
            if constexpr (kSelf) ri = self_eligible(ri, self.row0 + rec.row, self.mode) ? ri : -1;
            float a_acc = 0.f, b_acc = 0.f;
            if (vec) {
                // eight float4 steps at a time, every load issued before the first FMA: the rows come out of L2 (~600 cycles).
                // (A software pipeline across batches -- next batch's loads before this batch's FMAs -- was measured: nothing at
                // BASELINE configs[1], where the phase is latency-bound but runs beside the others, and 4 % SLOWER with a million
                // records, where sixteen warps per SM hide the latency and the register copies are pure cost.)
                const float4* c4 = reinterpret_cast<const float4*>(c_smem);
                const float4* r4 = reinterpret_cast<const float4*>(ref + (ri >= 0 ? ri : 0) * dim);
                const int nq = dim >> 2;
                constexpr int kU = 8;
                for (int q0 = sub; q0 < nq; q0 += kU * L) {
                    float4 rv[kU];
#pragma unroll
                    for (int u = 0; u < kU; ++u)
                        rv[u] = (ri >= 0 && q0 + u * L < nq) ? __ldg(r4 + q0 + u * L) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int u = 0; u < kU; ++u) {
                        const float4 cv = q0 + u * L < nq ? c4[q0 + u * L] : make_float4(0.f, 0.f, 0.f, 0.f);
                        a_acc = fmaf(cv.x, rv[u].x, a_acc); a_acc = fmaf(cv.y, rv[u].y, a_acc);
                        a_acc = fmaf(cv.z, rv[u].z, a_acc); a_acc = fmaf(cv.w, rv[u].w, a_acc);
                        b_acc = fmaf(rv[u].x, rv[u].x, b_acc); b_acc = fmaf(rv[u].y, rv[u].y, b_acc);
                        b_acc = fmaf(rv[u].z, rv[u].z, b_acc); b_acc = fmaf(rv[u].w, rv[u].w, b_acc);
                    }
                }
            } else {
                for (int q = sub; q < dim; q += L) {
                    const float rvq = ri >= 0 ? __ldg(ref + ri * dim + q) : 0.f;
                    a_acc = fmaf(c_smem[q], rvq, a_acc);
                    b_acc = fmaf(rvq, rvq, b_acc);
                }
            }
            for (int o = L >> 1; o > 0; o >>= 1) {                // the L lanes of a reference hold partial sums
                a_acc += __shfl_xor_sync(0xffffffffu, a_acc, o);
                b_acc += __shfl_xor_sync(0xffffffffu, b_acc, o);
            }
            // NOTE: the accumulation order differs from cos_fp32's lane-strided one by fp32 summation noise only (<= ~1e-7); the
            // decision between references that close is fp32-ill-defined anyway (tests: TIE_EPS)
            if (ri >= 0) {
                const float sc = __fdiv_rn(a_acc, __fmul_rn(__fsqrt_rn(b_acc), cc_sqrt));
                const unsigned long long kj = pack_key(sc, static_cast<int32_t>(ri));
                key = kj > key ? kj : key;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
            key = other > key ? other : key;
        }
        if (lane == 0) {
            float v;
            int32_t bi;
            unpack_key(key, v, bi);
            if (key == 0ull) { v = -INFINITY; bi = 0; }
            emit_result(rec.row, v, bi, thr, ref_index_base, keep, best_idx, best_val, band_tol, band_count, band_rows, band_cap);
        }
    }
}

// Work items are (group of kFullGroup flagged rows, slice of kSliceRefs references), handed out round-robin over a
// fixed grid (the flagged-row count only exists on the device); n_slices slices merge into one result per row.
constexpr int kSliceRefs = 1024;

// K3b, few rows: when (flagged rows x references) is small the tiled walk below is pure latency (one block crawls through
// a whole 1024-reference slice for a handful of rows: ~25 us at 1k references).  Here every warp of the grid takes
// (row, block of kSmallRefs references) items instead: the row is parked in this warp's shared-memory slot, lanes split
// the embedding, one fp32 cosine per reference exactly like K3a (kSmallBatch references in flight).  Same merge: atomicMax on the packed key, and the
// last item of a group of kFullGroup rows (full_ctr counts rows x blocks) writes the group's outputs.
constexpr int kSmallRefs = 8;        // one batch per item: with a handful of rows (BASELINE configs[1]: 2 of 100 k) the phase is pure
constexpr int kSmallBatch = 8;       // latency, and 32-reference items meant four dependent L2 round trips per warp (8 -> 3 us)
// every flagged row streams the whole reference set once here (no reuse across rows, unlike the tiled walk's 8 rows per
// reference read): only worth it while that is a few tens of MB of L2 traffic
constexpr long long kSmallElems = 16000000;

// (runs are dealt starting in the MIDDLE of the grid: away from the warps that hold the first pair and part records)
__device__ __forceinline__ int64_t small_first_item(int64_t warp, int64_t nwarps, int64_t ipw) {
    const int64_t half = nwarps >> 1;
    return (warp >= half ? warp - half : warp + (nwarps - half)) * ipw;
}

// kSelf: the per-candidate bound (!= g, or < g) is applied before the comparison
template <bool kSelf>
__device__ __forceinline__ void
rescan_small_phase(float* s_rows, const float* __restrict__ ref, int64_t n_ref, const float* __restrict__ cand, int32_t dim,
                   float thr, int64_t ref_index_base, uint8_t* __restrict__ keep, int32_t* __restrict__ best_idx,
                   float* __restrict__ best_val, const RecheckLists& lists, int64_t count, float band_tol,
                   int32_t* band_count, int64_t* band_rows, int64_t band_cap, bool vec, int emode, SelfArgs self) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    float* c_smem = s_rows + static_cast<size_t>(w) * dim;
    const int64_t nb = (n_ref + kSmallRefs - 1) / kSmallRefs;
    const int64_t n_items = count * nb;
    const int64_t warp = static_cast<int64_t>(blockIdx.x) * kWarps + w;
    const int64_t nwarps = static_cast<int64_t>(gridDim.x) * kWarps;
    // every warp takes a CONTIGUOUS run of items: consecutive reference blocks of the same row, so the row is parked once
    // and the warp merges its blocks in registers -- one atomicMax + one counter update per (warp, row), not per item
    const int64_t ipw = (n_items + nwarps - 1) / nwarps;
    const int64_t i0 = small_first_item(warp, nwarps, ipw);
    const int64_t i1 = (i0 + ipw < n_items) ? i0 + ipw : n_items;
    int64_t cur = -1;
    int32_t pending = 0;
    float cc_sqrt = 0.f, best = -INFINITY;
    int32_t bi = 0x7FFFFFFF;
    auto flush = [&]() {
        if (cur < 0 || pending == 0) return;
        if (lane == 0 && bi != 0x7FFFFFFF) atomicMax(&lists.full_keys[cur], pack_key(best, bi));
        __threadfence();
        const int64_t g = cur / kFullGroup;
        const int64_t rows_in_g = (count - g * kFullGroup < kFullGroup) ? count - g * kFullGroup : kFullGroup;
        int last = 0;
        if (lane == 0) last = (atomicAdd(&lists.full_ctr[g], pending) + pending == static_cast<int>(rows_in_g * nb)) ? 1 : 0;
        last = __shfl_sync(0xffffffffu, last, 0);
        if (last && lane < rows_in_g) {                          // every block of every row of the group has been merged
            __threadfence();
            const int64_t sl = g * kFullGroup + lane;
            const unsigned long long key = atomicAdd(&lists.full_keys[sl], 0ull);      // coherent read
            float v;
            int32_t bidx;
            unpack_key(key, v, bidx);
            if (key == 0ull) { v = -INFINITY; bidx = 0; }
            if (emode >= 0) best_idx[lists.full_rows[sl]] = static_cast<int32_t>(bidx + ref_index_base);
            else emit_result(lists.full_rows[sl], v, bidx, thr, ref_index_base, keep, best_idx, best_val, band_tol,
                             band_count, band_rows, band_cap);
        }
    };
    if (emode >= 0) {           // Euclid: score = -distance, so the key's "largest, then smallest index" is the first argmin
        for (int64_t item = i0; item < i1; ++item) {
            const int64_t slot = item / nb, blk = item - slot * nb;
            if (slot != cur) { flush(); cur = slot; pending = 0; best = -INFINITY; bi = 0x7FFFFFFF; }
            const int32_t crow = lists.full_rows[slot];
            const float* c = cand + static_cast<int64_t>(crow) * dim;
            const int64_t lo = blk * kSmallRefs, hi = (lo + kSmallRefs < n_ref) ? lo + kSmallRefs : n_ref;
            for (int64_t i = lo; i < hi; ++i) {
                if constexpr (kSelf) { if (!self_eligible(i, self.row0 + crow, self.mode)) continue; }
                const float sc = -k2s_euclid_dist(c, ref + i * dim, dim, lane, emode);
                if (sc > best) { best = sc; bi = static_cast<int32_t>(i); }
            }
            ++pending;
        }
        flush();
        return;
    }
    const int nvec = dim >> 2;
    if (vec && nvec <= 32) {
        // rows of <= 128 floats: one float4 per lane and row, all in registers, and the item's reference rows (which need no
        // list entry to be named) are requested BEFORE the candidate row's index is even known -- the phase is a chain of
        // memory latencies.  Same arithmetic as cos_fp32, bit for bit.
        static_assert(kSmallRefs == kSmallBatch, "one batch per item");
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4* ref4 = reinterpret_cast<const float4*>(ref);
        const bool live = lane < nvec;
        float4 cv = z4;
        int64_t g_self = 0;                                        // kSelf: global index of the parked row
        for (int64_t item = i0; item < i1; ++item) {
            const int64_t slot = item / nb, blk = item - slot * nb;
            const int64_t lo = blk * kSmallRefs;
            const int n_rows = static_cast<int>(n_ref - lo < kSmallRefs ? n_ref - lo : kSmallRefs);
            float4 rv[kSmallBatch];
#pragma unroll
            for (int r = 0; r < kSmallBatch; ++r)
                rv[r] = live ? __ldg(ref4 + (lo + (r < n_rows ? r : n_rows - 1)) * nvec + lane) : z4;
            if (slot != cur) {
                flush();
                cv = live ? __ldg(reinterpret_cast<const float4*>(cand) + static_cast<int64_t>(lists.full_rows[slot]) * nvec + lane) : z4;
                if constexpr (kSelf) g_self = self.row0 + lists.full_rows[slot];
                float cc = 0.f;
                cc = fmaf(cv.x, cv.x, cc); cc = fmaf(cv.y, cv.y, cc); cc = fmaf(cv.z, cv.z, cc); cc = fmaf(cv.w, cv.w, cc);
                cc_sqrt = __fsqrt_rn(warp_sum(cc));
                cur = slot;
                pending = 0;
                best = -INFINITY;
                bi = 0x7FFFFFFF;
            }
            float a[kSmallBatch], b[kSmallBatch];
#pragma unroll
            for (int r = 0; r < kSmallBatch; ++r) {
                a[r] = 0.f; b[r] = 0.f;
                a[r] = fmaf(cv.x, rv[r].x, a[r]); a[r] = fmaf(cv.y, rv[r].y, a[r]);
                a[r] = fmaf(cv.z, rv[r].z, a[r]); a[r] = fmaf(cv.w, rv[r].w, a[r]);
                b[r] = fmaf(rv[r].x, rv[r].x, b[r]); b[r] = fmaf(rv[r].y, rv[r].y, b[r]);
                b[r] = fmaf(rv[r].z, rv[r].z, b[r]); b[r] = fmaf(rv[r].w, rv[r].w, b[r]);
            }
#pragma unroll
            for (int r = 0; r < kSmallBatch; ++r) { a[r] = warp_sum(a[r]); b[r] = warp_sum(b[r]); }
#pragma unroll
            for (int r = 0; r < kSmallBatch; ++r) {              // ascending + strict '>' = first occurrence
                const float sc = __fdiv_rn(a[r], __fmul_rn(__fsqrt_rn(b[r]), cc_sqrt));
                if (r < n_rows && sc > best && (!kSelf || self_eligible(lo + r, g_self, self.mode))) { best = sc; bi = static_cast<int32_t>(lo + r); }
            }
            ++pending;
        }
        flush();
        return;
    }
    int64_t g_self = 0;
    for (int64_t item = i0; item < i1; ++item) {
        const int64_t slot = item / nb, blk = item - slot * nb;
        if (slot != cur) {
            flush();
            if constexpr (kSelf) g_self = self.row0 + lists.full_rows[slot];
            const float* c = cand + static_cast<int64_t>(lists.full_rows[slot]) * dim;
            float cc = 0.f;
            __syncwarp();
            for (int d = lane; d < dim; d += 32) { const float t = __ldg(c + d); c_smem[d] = t; cc = fmaf(t, t, cc); }
            __syncwarp();
            cc_sqrt = __fsqrt_rn(warp_sum(cc));
            cur = slot;
            pending = 0;
            best = -INFINITY;
            bi = 0x7FFFFFFF;
        }
        const int64_t lo = blk * kSmallRefs;
        const int64_t hi = (lo + kSmallRefs < n_ref) ? lo + kSmallRefs : n_ref;
        for (int64_t i = lo; i < hi; i += kSmallBatch) {         // ascending + strict '>' = first occurrence
            float sc[kSmallBatch];
            const int n_rows = static_cast<int>(hi - i < kSmallBatch ? hi - i : kSmallBatch);
            cos_fp32_multi<kSmallBatch>(c_smem, ref + i * dim, n_rows, dim, cc_sqrt, lane, vec, sc);
#pragma unroll
            for (int r = 0; r < kSmallBatch; ++r)
                if (r < n_rows && sc[r] > best && (!kSelf || self_eligible(i + r, g_self, self.mode))) { best = sc[r]; bi = static_cast<int32_t>(i + r); }
        }
        ++pending;
    }
    flush();
}

// One launch re-checks everything K2 flagged: phase A = K3a (pairs list), phase B = K3b (full-rescan list; small or
// tiled walk, chosen from the device-side count, uniform over the grid).  The phases touch disjoint rows.
// kSelf (ffr_filter_self): cand = rows [self.row0, ...) of ref; the pairs phase needs nothing (its leading references come from
// K2's masked scores), the parts phase and both full-rescan walks skip the references the row may not match.
template <bool kVec, bool kEuclid, bool kSelf = false>
__global__ void __launch_bounds__(kThreads, 2)      // two CTAs per SM (<= 128 registers): the fixed grid of 2 x SMs is ONE wave
recheck_kernel(const float* __restrict__ ref, int64_t n_ref, const float* __restrict__ cand, int32_t dim, float thr,
               int64_t ref_index_base, uint8_t* __restrict__ keep, int32_t* __restrict__ best_idx,
               float* __restrict__ best_val, RecheckLists lists, float band_tol, int32_t* band_count,
               int64_t* band_rows, int64_t band_cap, const int32_t* __restrict__ ref_map,
               const int32_t* __restrict__ n_unique_dev, int emode_arg, SelfArgs self) {
    const int emode = kEuclid ? emode_arg : -1;           // K2s distance mode (Euclid), -1 = cosine
    extern __shared__ __align__(16) float s_c[];               // kFullGroup x dim candidate rows | staged reference tile
    __shared__ float s_ccs[kFullGroup];
    __shared__ unsigned long long s_key[kWarps][kFullGroup];
    __shared__ int s_last;
    __shared__ int64_t s_g[kSelf ? kFullGroup : 1];           // kSelf: global indices of the parked full-rescan rows
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    recheck_pairs_phase(s_c, ref, cand, dim, thr, ref_index_base, keep, best_idx, best_val, lists, band_tol, band_count,
                        band_rows, band_cap, kVec, emode);
    recheck_parts_phase<kSelf>(s_c, ref, n_ref, cand, dim, thr, ref_index_base, keep, best_idx, best_val, lists, band_tol,
                               band_count, band_rows, band_cap, kVec, ref_map, n_unique_dev, emode, self);
    int64_t count = lists.hdr->full_count;
    if (count > lists.full_cap) count = lists.full_cap;
    if (count == 0) return;
    if (static_cast<long long>(count) * n_ref * dim <= kSmallElems) {
        rescan_small_phase<kSelf>(s_c, ref, n_ref, cand, dim, thr, ref_index_base, keep, best_idx, best_val, lists, count,
                                  band_tol, band_count, band_rows, band_cap, kVec, emode, self);
        return;
    }
    __syncthreads();                                            // phase A's per-warp rows are dead: the tiled walk reuses s_c
    // duplicate references folded before K2 (ref_map: compact column -> original row, ascending): the walk visits the UNIQUE
    // rows only -- a later bit-identical copy can never be the first occurrence of the maximum -- and works on compact
    // indices (their order is the original order), mapped back when a row's result is written
    const int64_t n_walk = n_unique_dev != nullptr ? static_cast<int64_t>(__ldg(n_unique_dev)) : n_ref;
    const int64_t n_slices = (n_walk + kSliceRefs - 1) / kSliceRefs;
    const int64_t n_groups = (count + kFullGroup - 1) / kFullGroup;
    const int64_t n_items = n_groups * n_slices;
    int64_t parked = -1;
    for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int64_t g = item / n_slices, slice = item - g * n_slices;
        const int64_t lo = slice * kSliceRefs;
        const int64_t hi = (lo + kSliceRefs < n_walk) ? lo + kSliceRefs : n_walk;
        __syncthreads();
        if (g != parked) {                                     // warp w parks candidate rows w, w + kWarps, ... of the group
            for (int jw = w; jw < kFullGroup; jw += kWarps) {
                const int64_t slot = g * kFullGroup + jw;
                float cc = 0.f;
                if (slot < count) {
                    // kVec: parked TRANSPOSED, [dim][kFullGroup] -- the sixteen candidates' values of one k are four float4, i.e.
                    // eight (candidate j, candidate j + 1) pairs for the packed FMAs below
                    const float* c = cand + static_cast<int64_t>(lists.full_rows[slot]) * dim;
                    for (int d = lane; d < dim; d += 32) {
                        const float t = __ldg(c + d);
                        s_c[kVec ? d * kFullGroup + jw : jw * dim + d] = t;
                        cc = fmaf(t, t, cc);
                    }
                } else {
                    for (int d = lane; d < dim; d += 32) s_c[kVec ? d * kFullGroup + jw : jw * dim + d] = 0.f;
                }
                cc = warp_sum(cc);
                if (lane == 0) s_ccs[jw] = __fsqrt_rn(cc);
                if constexpr (kSelf) { if (lane == 0) s_g[jw] = slot < count ? self.row0 + lists.full_rows[slot] : 0; }
            }
            parked = g;
        }
        __syncthreads();
        float best[kFullGroup];
        int32_t bidx[kFullGroup];
#pragma unroll
        for (int j = 0; j < kFullGroup; ++j) { best[j] = -INFINITY; bidx[j] = 0x7FFFFFFF; }
        if (kVec) {
            // References are staged through shared memory in [kTileRefs refs] x [kKC floats] tiles (row stride kKCPad
            // floats: the float4 reads of 8 consecutive threads hit 8 disjoint bank groups), the next tile chunk is
            // prefetched into registers while the current one is consumed, and every thread owns a register tile of
            // kRefsPerThread references (t, t + 256, ...) x kFullGroup candidates: per 8 K-values it issues 8 + 16
            // shared loads for 256 FMAs (the candidate loads are warp-wide broadcasts).
            // (round 2: the tiles go global -> shared with cp.async into TWO buffers -- no staging registers, no shared-memory
            // stores by the threads, one barrier per chunk instead of two)
            float* s_r0 = s_c + kFullGroup * dim;
            constexpr int kTileFloats = kTileRefs * kKCPad;
            const int n_kc = (dim + kKC - 1) / kKC;
            const int64_t n_rt = (hi - lo + kTileRefs - 1) / kTileRefs;
            const int64_t n_it = n_rt * n_kc;
            constexpr int kPf = kTileRefs * (kKC / 4) / kThreads;          // 16-byte pieces per thread per chunk (8)
            int64_t rowi[kPf];                                             // the rows this thread copies from, per reference tile
            auto fetch = [&](int64_t rt, int kc, int buf) {
                const int64_t i0 = lo + rt * kTileRefs;
                float* dst = s_r0 + buf * kTileFloats;
                if (kc == 0) {
#pragma unroll
                    for (int u = 0; u < kPf; ++u) {
                        const int64_t gi = i0 + ((threadIdx.x + kThreads * u) >> 1);
                        rowi[u] = gi < hi ? (ref_map != nullptr ? static_cast<int64_t>(__ldg(ref_map + gi)) : gi) : -1;
                    }
                }
#pragma unroll
                for (int u = 0; u < kPf; ++u) {
                    const int f = threadIdx.x + kThreads * u;              // 2 float4 per reference row
                    const int col = kc * kKC + (f & 1) * 4;
                    const bool ok = rowi[u] >= 0 && col < dim;
                    // (src-size 0 = the 16 bytes are zero-filled: rows past the slice, columns past dim)
                    const float* src = ok ? ref + rowi[u] * dim + col : ref;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;"
                                 ::"r"(smem_u32(dst + (f >> 1) * kKCPad + (f & 1) * 4)), "l"(src), "r"(ok ? 16 : 0) : "memory");
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
            };
            fetch(0, 0, 0);
            // accumulators as (candidate 2p, candidate 2p + 1) pairs: one FFMA2 (sm_100 packed fp32) per pair and k -- the same
            // IEEE fma per candidate, in the same order over k, at half the FMA-pipe instructions (the walk is FMA-issue-bound)
            static_assert(kFullGroup == 16, "four float4 of candidates per k");
            float2 acc[kRefsPerThread][kFullGroup / 2];
            float rr[kRefsPerThread];
            int64_t rt = 0;
            int kc = 0;
            for (int64_t it = 0; it < n_it; ++it) {
                if (kc == 0) {
#pragma unroll
                    for (int r = 0; r < kRefsPerThread; ++r) {
                        rr[r] = 0.f;
#pragma unroll
                        for (int j = 0; j < kFullGroup / 2; ++j) acc[r][j] = make_float2(0.f, 0.f);
                    }
                }
                asm volatile("cp.async.wait_group 0;" ::: "memory");     // this thread's pieces of chunk `it` have landed ...
                __syncthreads();                                         // ... everybody's have, and chunk it - 1 has been consumed
                const float* s_r = s_r0 + static_cast<int>(it & 1) * kTileFloats;
                int nkc = kc + 1;
                int64_t nrt = rt;
                if (nkc == n_kc) { nkc = 0; ++nrt; }
                if (it + 1 < n_it) fetch(nrt, nkc, static_cast<int>((it + 1) & 1));   // in flight while this chunk is consumed
#pragma unroll
                for (int j4 = 0; j4 < kKC / 4; ++j4) {
                    const int col = kc * kKC + j4 * 4;
                    if (col < dim) {
                        float rv[kRefsPerThread][4];
#pragma unroll
                        for (int r = 0; r < kRefsPerThread; ++r) {
                            const float4 t = *reinterpret_cast<const float4*>(s_r + (threadIdx.x + r * kThreads) * kKCPad + j4 * 4);
                            rv[r][0] = t.x; rv[r][1] = t.y; rv[r][2] = t.z; rv[r][3] = t.w;
                            if (!kEuclid) {
                                rr[r] = fmaf(t.x, t.x, rr[r]); rr[r] = fmaf(t.y, t.y, rr[r]);
                                rr[r] = fmaf(t.z, t.z, rr[r]); rr[r] = fmaf(t.w, t.w, rr[r]);
                            }
                        }
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            float2 cp[kFullGroup / 2];
#pragma unroll
                            for (int q4 = 0; q4 < kFullGroup / 4; ++q4) {
                                const float4 c4 = *reinterpret_cast<const float4*>(s_c + (col + kk) * kFullGroup + q4 * 4);
                                cp[2 * q4] = make_float2(c4.x, c4.y);
                                cp[2 * q4 + 1] = make_float2(c4.z, c4.w);
                            }
#pragma unroll
                            for (int r = 0; r < kRefsPerThread; ++r) {
                                const float2 r2 = make_float2(rv[r][kk], rv[r][kk]);
                                if (kEuclid) {                  // d = c - r (one rounding, as a subtraction), then d * d
                                    const float2 m1 = make_float2(-1.0f, -1.0f);
#pragma unroll
                                    for (int pj = 0; pj < kFullGroup / 2; ++pj) {
                                        const float2 d = __ffma2_rn(r2, m1, cp[pj]);
                                        acc[r][pj] = __ffma2_rn(d, d, acc[r][pj]);
                                    }
                                } else {
#pragma unroll
                                    for (int pj = 0; pj < kFullGroup / 2; ++pj) acc[r][pj] = __ffma2_rn(cp[pj], r2, acc[r][pj]);
                                }
                            }
                        }
                    }
                }
                if (kc == n_kc - 1) {
#pragma unroll
                    for (int r = 0; r < kRefsPerThread; ++r) {                    // ascending reference index per thread
                        const int64_t i = lo + rt * kTileRefs + threadIdx.x + r * kThreads;
                        if (i < hi) {
                            const float rs = __fsqrt_rn(rr[r]);
#pragma unroll
                            for (int j = 0; j < kFullGroup; ++j) {
                                const float dot = (j & 1) ? acc[r][j >> 1].y : acc[r][j >> 1].x;
                                const float sc = kEuclid ? -__fsqrt_rn(dot) : __fdiv_rn(dot, __fmul_rn(rs, s_ccs[j]));
                                if (sc > best[j] && (!kSelf || self_eligible(i, s_g[j], self.mode))) { best[j] = sc; bidx[j] = static_cast<int32_t>(i); }
                            }
                        }
                    }
                }
                kc = nkc;
                rt = nrt;
            }
        } else {
            for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) {
                float acc[kFullGroup];
#pragma unroll
                for (int j = 0; j < kFullGroup; ++j) acc[j] = 0.f;
                float rr = 0.f;
                const float* r = ref + (ref_map != nullptr ? static_cast<int64_t>(__ldg(ref_map + i)) : i) * dim;
                for (int k = 0; k < dim; ++k) {
                    const float rv = __ldg(r + k);
                    rr = fmaf(rv, rv, rr);
#pragma unroll
                    for (int j = 0; j < kFullGroup; ++j) {
                        if (kEuclid) { const float d = s_c[j * dim + k] - rv; acc[j] = fmaf(d, d, acc[j]); }
                        else acc[j] = fmaf(s_c[j * dim + k], rv, acc[j]);
                    }
                }
                const float rs = __fsqrt_rn(rr);
#pragma unroll
                for (int j = 0; j < kFullGroup; ++j) {
                    const float sc = kEuclid ? -__fsqrt_rn(acc[j]) : __fdiv_rn(acc[j], __fmul_rn(rs, s_ccs[j]));
                    if (sc > best[j] && (!kSelf || self_eligible(i, s_g[j], self.mode))) { best[j] = sc; bidx[j] = static_cast<int32_t>(i); }
                }
            }
        }
        // block merge: warp shuffle max on the packed key, then one atomicMax per row
#pragma unroll
        for (int j = 0; j < kFullGroup; ++j) {
            unsigned long long key = (bidx[j] == 0x7FFFFFFF) ? 0ull : pack_key(best[j], bidx[j]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
                key = other > key ? other : key;
            }
            if (lane == 0) s_key[w][j] = key;
        }
        __syncthreads();
        if (threadIdx.x < kFullGroup) {
            const int j = threadIdx.x;
            unsigned long long key = 0ull;
            for (int ww = 0; ww < kWarps; ++ww) key = s_key[ww][j] > key ? s_key[ww][j] : key;
            const int64_t slot = g * kFullGroup + j;
            if (slot < count && key != 0ull) atomicMax(&lists.full_keys[slot], key);
        }
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_last = (atomicAdd(&lists.full_ctr[g], 1) == static_cast<int>(n_slices) - 1) ? 1 : 0;
        __syncthreads();
        if (s_last && threadIdx.x < kFullGroup) {
            __threadfence();
            const int64_t slot = g * kFullGroup + threadIdx.x;
            if (slot < count) {
                const unsigned long long key = atomicAdd(&lists.full_keys[slot], 0ull);     // coherent read
                float v;
                int32_t bi;
                unpack_key(key, v, bi);
                if (key == 0ull) { v = -INFINITY; bi = 0; }
                else if (ref_map != nullptr) bi = __ldg(ref_map + bi);          // compact column -> original reference
                if (kEuclid) best_idx[lists.full_rows[slot]] = static_cast<int32_t>(bi + ref_index_base);
                else emit_result(lists.full_rows[slot], v, bi, thr, ref_index_base, keep, best_idx, best_val, band_tol,
                                 band_count, band_rows, band_cap);
            }
        }
    }
}

// packed per-rank record block for the allgather: [idx i32 x m_pad][keep u8 x m_pad], m_pad = m rounded up to 16
__global__ void pack_results_kernel(const uint8_t* __restrict__ keep, const int32_t* __restrict__ idx, int64_t m,
                                    int64_t m_pad, uint8_t* __restrict__ packed) {
    int32_t* pidx = reinterpret_cast<int32_t*>(packed);
    uint8_t* pkeep = packed + m_pad * 4;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < m;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        pidx[i] = idx[i];
        pkeep[i] = keep[i];
    }
}

__global__ void unpack_results_kernel(const uint8_t* __restrict__ packed, int64_t m, int64_t m_pad, int nranks,
                                      uint8_t* __restrict__ keep, int32_t* __restrict__ idx) {
    const int64_t total = m * nranks;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t r = i / m, j = i - r * m;
        const uint8_t* blk = packed + r * m_pad * 5;
        idx[i] = reinterpret_cast<const int32_t*>(blk)[j];
        keep[i] = blk[m_pad * 4 + j];
    }
}

// |c| of one candidate row, lane-strided (float4 #(lane + 32 j) when vec), warp_sum, IEEE sqrt: the norm the all-reduce merge
// and the match lists hand cos_fp32.  The whole warp calls it; every lane returns the norm.
__device__ __forceinline__ float cand_norm_fp32(const float* __restrict__ c, int32_t dim, int lane, bool vec) {
    float cc = 0.f;
    if (vec) {
        const float4* c4 = reinterpret_cast<const float4*>(c);
        for (int k = lane; k < (dim >> 2); k += 32) {
            const float4 t = __ldg(c4 + k);
            cc = fmaf(t.x, t.x, cc); cc = fmaf(t.y, t.y, cc); cc = fmaf(t.z, t.z, cc); cc = fmaf(t.w, t.w, cc);
        }
    } else {
        for (int d = lane; d < dim; d += 32) { const float t = __ldg(c + d); cc = fmaf(t, t, cc); }
    }
    return __fsqrt_rn(warp_sum(cc));
}

// ---- gallery over ranks (ffr_allreduce_best) --------------------------------------------------------------------------
// Merge / value pass: the fp32 value of each row's winner on this rank, packed into the merge key with pack_key (above) --
// (orderable(v) << 32) | ~global_idx, v = cosine score or -distance, so "largest key" = best value, then smallest global index
// (the first occurrence, np.argmax / np.argmin over the whole gallery).  Key 0 is the identity: a rank without references, or
// a row whose index lies outside this rank's shard, contributes nothing.  Cosine uses K3's fp32 arithmetic (cos_fp32 on the
// row's own |c|, lane-strided as in the parked-row form), Euclid K2s's (k2s_euclid_dist in mode emode), so that a rank's value
// equals what the one-GPU call computes for that same pair.  One warp per row.
__global__ void __launch_bounds__(kThreads)
best_key_kernel(const float* __restrict__ ref, int64_t n_ref, int64_t ref_index_base, const float* __restrict__ cand,
                int64_t n_cand, int32_t dim, const int32_t* __restrict__ best_idx, unsigned long long* __restrict__ keys,
                bool vec, int emode) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = static_cast<int64_t>(blockIdx.x) * kWarps + (threadIdx.x >> 5);
    const int64_t nwarps = static_cast<int64_t>(gridDim.x) * kWarps;
    for (int64_t row = warp; row < n_cand; row += nwarps) {
        const int32_t g = __ldg(best_idx + row);
        const int64_t ri = static_cast<int64_t>(g) - ref_index_base;
        if (ri < 0 || ri >= n_ref) {
            if (lane == 0) keys[row] = 0ull;
            continue;
        }
        const float* c = cand + row * dim;
        const float* r = ref + ri * dim;
        float v;
        if (emode >= 0) {
            v = -k2s_euclid_dist(c, r, dim, lane, emode);
        } else {
            v = cos_fp32(c, r, dim, cand_norm_fp32(c, dim, lane, vec), lane, vec);
        }
        if (lane == 0) keys[row] = pack_key(v, g);
    }
}

// After the all-reduce: global best_idx / best_val, keep from thr and the band, from the winning key.  A row no rank had a
// reference for (key 0) gets keep 0, index -1 and -inf (cosine) / +inf (Euclid), never in the band.
__global__ void emit_keys_kernel(const unsigned long long* __restrict__ keys, int64_t n_cand, bool euclid, float thr,
                                 uint8_t* __restrict__ keep, int32_t* __restrict__ best_idx, float* __restrict__ best_val,
                                 float band_tol, int32_t* band_count, int64_t* band_rows, int64_t band_cap) {
    for (int64_t row = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; row < n_cand;
         row += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const unsigned long long k = keys[row];
        if (k == 0ull) {
            keep[row] = 0;
            best_idx[row] = -1;
            if (best_val != nullptr) best_val[row] = euclid ? INFINITY : -INFINITY;
            continue;
        }
        float v;
        int32_t g;
        unpack_key(k, v, g);
        const float best = euclid ? -v : v;
        keep[row] = (euclid ? best <= thr : best >= thr) ? 1 : 0;
        best_idx[row] = g;
        if (best_val != nullptr) best_val[row] = best;
        if (band_count != nullptr && fabsf(best - thr) <= band_tol) {
            const int32_t slot = atomicAdd(band_count, 1);
            if (band_rows != nullptr && slot < band_cap) band_rows[slot] = row;
        }
    }
}

// ---- match lists (ffr_match_pairs*) ---------------------------------------------------------------------------------------
// A pair's fp32 value, the contract's arithmetic on both paths: cosine = cos_fp32 on the candidate's cand_norm_fp32 (the merge's
// value), Euclid = k2s_euclid_dist in K2s's form emode.  c may be a parked copy of the candidate row: the arithmetic, not the
// address, fixes the bits.  The whole warp calls it; every lane returns the value.
template <bool kEuclid>
__device__ __forceinline__ float pair_value(const float* c, const float* __restrict__ r, int32_t dim, float c_norm, int lane,
                                            bool vec, int emode) {
    if constexpr (kEuclid) return k2s_euclid_dist(c, r, dim, lane, emode);
    else                   return cos_fp32(c, r, dim, c_norm, lane, vec);
}
template <bool kEuclid>
__device__ __forceinline__ bool pair_accepted(float v, float thr) { return kEuclid ? v <= thr : v >= thr; }

// Appends the warp's accepted pairs (lane k holds the k-th pair of this batch) with one atomic on *ctr; returns the batch's count
__device__ __forceinline__ uint32_t append_accepted(bool acc, int32_t row, int64_t ref, float v, unsigned long long* ctr,
                                                    const PairOut& out, int lane) {
    const uint32_t bal = __ballot_sync(0xffffffffu, acc);
    if (bal == 0u) return 0u;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(ctr, static_cast<unsigned long long>(__popc(bal)));
    base = __shfl_sync(0xffffffffu, base, 0);
    const unsigned long long slot = base + __popc(bal & ((1u << lane) - 1u));
    if (acc && slot < static_cast<unsigned long long>(out.cap)) {
        out.cand[slot] = row;
        out.ref[slot] = static_cast<int32_t>(ref);
        out.val[slot] = v;
    }
    return static_cast<uint32_t>(__popc(bal));
}

constexpr int kPairMaxDim = 512;      // the finishing pass runs behind the tensor-core path only (dim <= 512)

// Finishing pass.  Work items: groups of 32 raw entries (min(raw count, capacity) of them), then (exact row, 32 references).
// A warp takes a group's entries one after the other; K2 appends the columns of one (row, tile half) together, so the candidate
// row is parked in shared memory (and, cosine, its norm summed) once per run of entries, not once per entry.  Accepted pairs are
// appended warp-aggregated.  The last block to finish writes the caller's count: the accepted pairs, or when the raw list
// overflowed the raw count plus the exact rows' pairs (the accepted raw entries are a subset of the raw ones).
template <bool kEuclid>
__global__ void __launch_bounds__(kThreads)
pairs_finish_kernel(const float* __restrict__ ref, int64_t n_ref, const float* __restrict__ cand, int32_t dim, float thr,
                    int64_t ref_index_base, SelfArgs self, PairRaw raw, WsHeader* hdr, PairOut out, bool vec, int emode) {
    __shared__ __align__(16) float s_rows[kWarps][kPairMaxDim];
    const int lane = threadIdx.x & 31;
    float* c_s = s_rows[threadIdx.x >> 5];
    const int64_t warp = static_cast<int64_t>(blockIdx.x) * kWarps + (threadIdx.x >> 5);
    const int64_t nwarps = static_cast<int64_t>(gridDim.x) * kWarps;
    const unsigned long long raw_all = hdr->raw_count;
    const int64_t n_raw = raw_all < static_cast<unsigned long long>(raw.cap) ? static_cast<int64_t>(raw_all) : raw.cap;
    const int64_t n_exact = kEuclid ? hdr->exact_count : 0;
    const int64_t g_raw = (n_raw + 31) / 32, ref_chunks = (n_ref + 31) / 32;
    const int64_t n_items = g_raw + n_exact * ref_chunks;
    int64_t parked = -1;
    float c_norm = 0.f;
    const auto park = [&](int32_t row) {
        if (row == parked) return;
        const float* c = cand + static_cast<int64_t>(row) * dim;
        __syncwarp();
        for (int k = lane; k < dim; k += 32) c_s[k] = __ldg(c + k);
        __syncwarp();
        if (!kEuclid) c_norm = cand_norm_fp32(c, dim, lane, vec);
        parked = row;
    };
    for (int64_t it = warp; it < n_items; it += nwarps) {
        bool acc = false;
        int32_t my_row = 0;
        int64_t my_ref = 0;
        float my_v = 0.f;
        const bool exact = it >= g_raw;
        if (!exact) {
            const int64_t e = it * 32 + lane;
            const uint2 en = e < n_raw ? raw.raw[e] : make_uint2(0xFFFFFFFFu, 0u);
            for (int k = 0; k < 32; ++k) {
                const uint32_t row = __shfl_sync(0xffffffffu, en.x, k), col = __shfl_sync(0xffffffffu, en.y, k);
                if (row == 0xFFFFFFFFu) break;                                 // (the group's tail: the same for every lane)
                park(static_cast<int32_t>(row));
                const float v = pair_value<kEuclid>(c_s, ref + static_cast<int64_t>(col) * dim, dim, c_norm, lane, vec, emode);
                if (lane == k) { my_v = v; my_row = static_cast<int32_t>(row); my_ref = col; acc = pair_accepted<kEuclid>(v, thr); }
            }
        } else {
            const int64_t x = it - g_raw, i0 = (x % ref_chunks) * 32;
            const int32_t row = __ldg(raw.exact_rows + x / ref_chunks);
            park(row);
            const int64_t i_end = self.mode >= 0 ? (self.row0 + row < n_ref ? self.row0 + row : n_ref) : n_ref;
            for (int k = 0; k < 32 && i0 + k < i_end; ++k) {
                const float v = pair_value<kEuclid>(c_s, ref + (i0 + k) * dim, dim, c_norm, lane, vec, emode);
                if (lane == k) { my_v = v; my_row = row; my_ref = i0 + k; acc = pair_accepted<kEuclid>(v, thr); }
            }
        }
        const uint32_t n_acc = append_accepted(acc, my_row, my_ref + ref_index_base, my_v, &hdr->acc_count, out, lane);
        if (exact && n_acc != 0u && lane == 0) atomicAdd(&hdr->acc_exact, static_cast<unsigned long long>(n_acc));
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(&hdr->pairs_blocks, 1) == static_cast<int32_t>(gridDim.x) - 1) {
        __threadfence();
        const unsigned long long acc = atomicAdd(&hdr->acc_count, 0ull), ex = atomicAdd(&hdr->acc_exact, 0ull);
        *out.count = static_cast<int64_t>(raw_all > static_cast<unsigned long long>(raw.cap) ? raw_all + ex : acc);
    }
}

// Exact path: one warp per candidate row against every reference (self: the rows i < g), 32 references per append
template <bool kEuclid>
__global__ void __launch_bounds__(kThreads)
pairs_exact_kernel(const float* __restrict__ ref, int64_t n_ref, const float* __restrict__ cand, int64_t n_cand, int32_t dim,
                   float thr, int64_t ref_index_base, SelfArgs self, PairOut out, bool vec, int emode) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = static_cast<int64_t>(blockIdx.x) * kWarps + (threadIdx.x >> 5);
    const int64_t nwarps = static_cast<int64_t>(gridDim.x) * kWarps;
    unsigned long long* ctr = reinterpret_cast<unsigned long long*>(out.count);
    for (int64_t row = warp; row < n_cand; row += nwarps) {
        const float* c = cand + row * dim;
        const float c_norm = kEuclid ? 0.f : cand_norm_fp32(c, dim, lane, vec);
        const int64_t i_end = self.mode >= 0 ? (self.row0 + row < n_ref ? self.row0 + row : n_ref) : n_ref;
        for (int64_t i0 = 0; i0 < i_end; i0 += 32) {
            bool acc = false;
            float my_v = 0.f;
            for (int k = 0; k < 32 && i0 + k < i_end; ++k) {
                const float v = pair_value<kEuclid>(c, ref + (i0 + k) * dim, dim, c_norm, lane, vec, emode);
                if (lane == k) { my_v = v; acc = pair_accepted<kEuclid>(v, thr); }
            }
            append_accepted(acc, static_cast<int32_t>(row), i0 + lane + ref_index_base, my_v, ctr, out, lane);
        }
    }
}

// the candidates' float4 form (cos_fp32 / cand_norm_fp32) and K2s's Euclid form, the same for both paths of a call
bool pairs_vec(const float* ref, const float* cand, int32_t dim) {
    return (dim % 4 == 0) && ((reinterpret_cast<uintptr_t>(ref) & 15) == 0) && ((reinterpret_cast<uintptr_t>(cand) & 15) == 0);
}
int pairs_emode(const float* ref, const float* cand, int64_t n_ref, int32_t dim, int metric, SelfArgs self) {
    if (metric != FFR_METRIC_EUCLID) return -1;
    return k2s_form(ref, cand, self.mode >= 0 ? INT64_MAX : n_ref, dim);
}

}  // namespace

int launch_pairs_finish(const float* ref, int64_t n_ref, const float* cand, int32_t dim, int metric, float thr, int64_t ref_index_base,
                        SelfArgs self, const PairRaw& raw, WsHeader* hdr, const PairOut& out, cudaStream_t s) {
    if (dim > kPairMaxDim) { set_error("pairs: finishing pass needs dim <= %d", kPairMaxDim); return FFR_ERR_UNSUPPORTED; }
    const bool vec = pairs_vec(ref, cand, dim);
    const int emode = pairs_emode(ref, cand, n_ref, dim, metric, self);
    const unsigned grid = static_cast<unsigned>(num_sms()) * 4;
    if (emode >= 0) pairs_finish_kernel<true><<<grid, kThreads, 0, s>>>(ref, n_ref, cand, dim, thr, ref_index_base, self, raw, hdr, out, vec, emode);
    else            pairs_finish_kernel<false><<<grid, kThreads, 0, s>>>(ref, n_ref, cand, dim, thr, ref_index_base, self, raw, hdr, out, vec, emode);
    FFR_LAUNCH_CHECK("pairs_finish");
    return FFR_OK;
}

int launch_pairs_exact(const float* ref, int64_t n_ref, const float* cand, int64_t n_cand, int32_t dim, int metric, float thr,
                       int64_t ref_index_base, SelfArgs self, const PairOut& out, cudaStream_t s) {
    if (n_cand == 0) return FFR_OK;
    const bool vec = pairs_vec(ref, cand, dim);
    const int emode = pairs_emode(ref, cand, n_ref, dim, metric, self);
    int64_t grid = (n_cand + kWarps - 1) / kWarps;
    if (grid > static_cast<int64_t>(num_sms()) * 8) grid = static_cast<int64_t>(num_sms()) * 8;
    if (emode >= 0) pairs_exact_kernel<true><<<static_cast<unsigned>(grid), kThreads, 0, s>>>(ref, n_ref, cand, n_cand, dim, thr, ref_index_base, self, out, vec, emode);
    else            pairs_exact_kernel<false><<<static_cast<unsigned>(grid), kThreads, 0, s>>>(ref, n_ref, cand, n_cand, dim, thr, ref_index_base, self, out, vec, emode);
    FFR_LAUNCH_CHECK("pairs_exact");
    return FFR_OK;
}

int launch_best_keys(const float* ref, int64_t n_ref, int64_t ref_index_base, const float* cand, int64_t n_cand, int32_t dim,
                     int metric, const int32_t* best_idx, unsigned long long* keys, cudaStream_t s) {
    if (n_cand == 0) return FFR_OK;
    // K3's choice (launch_recheck) wherever K3 runs: its candidates are always 16-byte aligned there, these need not be
    const bool vec = (dim % 4 == 0) && ((reinterpret_cast<uintptr_t>(ref) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(cand) & 15) == 0);
    // the whole gallery's form (more than two references over all ranks): the merge reproduces the one-GPU call's values
    const int emode = metric == FFR_METRIC_EUCLID ? k2s_form(ref, cand, INT64_MAX, dim) : -1;
    int64_t grid = (n_cand + kWarps - 1) / kWarps;
    if (grid > static_cast<int64_t>(num_sms()) * 8) grid = static_cast<int64_t>(num_sms()) * 8;
    best_key_kernel<<<static_cast<unsigned>(grid), kThreads, 0, s>>>(ref, n_ref, ref_index_base, cand, n_cand, dim, best_idx,
                                                                      keys, vec, emode);
    FFR_LAUNCH_CHECK("best_keys");
    return FFR_OK;
}

int launch_emit_keys(const unsigned long long* keys, int64_t n_cand, int metric, float thr, const FilterOut& o, cudaStream_t s) {
    if (n_cand == 0) return FFR_OK;
    int64_t grid = (n_cand + 255) / 256;
    if (grid > static_cast<int64_t>(num_sms()) * 8) grid = static_cast<int64_t>(num_sms()) * 8;
    emit_keys_kernel<<<static_cast<unsigned>(grid), 256, 0, s>>>(keys, n_cand, metric == FFR_METRIC_EUCLID, thr, o.keep, o.idx,
                                                                o.val, o.band.tol, o.band.count, o.band.rows, o.band.cap);
    FFR_LAUNCH_CHECK("emit_keys");
    return FFR_OK;
}

int launch_recheck(const float* ref, int64_t n_ref, const float* cand, int64_t n_cand, int32_t dim, float thr,
                   int64_t ref_index_base, const FilterOut& o, RecheckLists lists, const int32_t* ref_map,
                   const int32_t* n_unique_dev, cudaStream_t s, int euclid_mode, SelfArgs self) {
    if (n_cand == 0) return FFR_OK;
    const bool euclid = euclid_mode >= 0;
    static_assert(kFullGroup % kWarps == 0, "every warp parks kFullGroup / kWarps candidate rows of a full-rescan group");
    const int sms = num_sms();
    // kFullGroup parked candidate rows (the per-warp phases use the first kWarps of them)
    const size_t smem = static_cast<size_t>(kFullGroup) * dim * sizeof(float);
    if (smem > 96 * 1024) { set_error("recheck: dim %d too large", dim); return FFR_ERR_UNSUPPORTED; }
    const int vec = (dim % 4 == 0) && ((reinterpret_cast<uintptr_t>(ref) & 15) == 0);
    // the flagged-row counts live on the device: ONE fixed grid strides over both lists (blocks without work exit at once)
    const int64_t gx = static_cast<int64_t>(sms) * 2;         // two blocks per SM are resident (registers): one wave
    const dim3 g2(static_cast<unsigned>(gx));
    const size_t smem_full = smem + 2 * static_cast<size_t>(kTileRefs) * kKCPad * sizeof(float);   // + two cp.async tile buffers
    {   // per-DEVICE function attribute: once for every device this process uses
        static std::mutex mu;
        static bool attr_set[kMaxDevices] = {};
        const int slot = current_device_slot();
        std::lock_guard<std::mutex> lock(mu);
        if (!attr_set[slot]) {
            FFR_CUDA_TRY(cudaFuncSetAttribute(recheck_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 148 * 1024));
            FFR_CUDA_TRY(cudaFuncSetAttribute(recheck_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 148 * 1024));
            FFR_CUDA_TRY(cudaFuncSetAttribute(recheck_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 148 * 1024));
            FFR_CUDA_TRY(cudaFuncSetAttribute(recheck_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 148 * 1024));
            FFR_CUDA_TRY(cudaFuncSetAttribute(recheck_kernel<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 148 * 1024));
            FFR_CUDA_TRY(cudaFuncSetAttribute(recheck_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 148 * 1024));
            FFR_CUDA_TRY(cudaFuncSetAttribute(recheck_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 148 * 1024));
            FFR_CUDA_TRY(cudaFuncSetAttribute(recheck_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 148 * 1024));
            attr_set[slot] = true;
        }
    }
    auto* fn = self.mode >= 0
                   ? (euclid ? (vec ? recheck_kernel<true, true, true> : recheck_kernel<false, true, true>)
                             : (vec ? recheck_kernel<true, false, true> : recheck_kernel<false, false, true>))
                   : (euclid ? (vec ? recheck_kernel<true, true> : recheck_kernel<false, true>)
                             : (vec ? recheck_kernel<true, false> : recheck_kernel<false, false>));
    fn<<<g2, kThreads, vec ? smem_full : smem, s>>>(ref, n_ref, cand, dim, thr, ref_index_base, o.keep, o.idx, o.val, lists,
                                                    o.band.tol, o.band.count, o.band.rows, o.band.cap, ref_map, n_unique_dev,
                                                    euclid_mode, self);
    FFR_LAUNCH_CHECK("recheck");
    return FFR_OK;
}

int launch_pack_results(const uint8_t* keep, const int32_t* idx, int64_t m, int64_t m_pad, uint8_t* packed,
                        cudaStream_t s) {
    if (m == 0) return FFR_OK;
    int64_t grid = (m + 255) / 256;
    if (grid > num_sms() * 8) grid = num_sms() * 8;
    pack_results_kernel<<<static_cast<unsigned>(grid), 256, 0, s>>>(keep, idx, m, m_pad, packed);
    FFR_LAUNCH_CHECK("pack_results");
    return FFR_OK;
}

int launch_unpack_results(const uint8_t* packed, int64_t m, int64_t m_pad, int nranks, uint8_t* keep, int32_t* idx,
                          cudaStream_t s) {
    if (m == 0) return FFR_OK;
    int64_t grid = (m * nranks + 255) / 256;
    if (grid > num_sms() * 8) grid = num_sms() * 8;
    unpack_results_kernel<<<static_cast<unsigned>(grid), 256, 0, s>>>(packed, m, m_pad, nranks, keep, idx);
    FFR_LAUNCH_CHECK("unpack_results");
    return FFR_OK;
}

}  // namespace ffr

// K2 -- fused reference x candidate cosine GEMM + threshold + running max/argmax, tcgen05/TMEM/TMA, sm_100a.
//
// Replaces the per-pair scan of
//     face_detection_and_extraction/face_extraction/extract_and_label_faces_from_dataset.py:101-116
// (cosine :106, threshold :110) and, through the unit-norm equivalence d <= t <=> cos >= 1 - t^2/2, the
// per-row test of similar_face_filtering/filter_faces_using_reference.py:186-189, for reference sets
// large enough to be tensor-core work.  The n_ref x n_cand similarity matrix only ever exists as
// 128 x 256 fp32 accumulator tiles in tensor memory; HBM sees the embeddings once and 9 bytes of result
// per candidate.
//
// Operands are the fp16, L2-normalised rows produced by K1 (leading dimension = dim rounded up to 64,
// zero padded), so the fp32 accumulator IS the cosine similarity.  fp16 operand rounding gives
// |score - fp32 score| ~ 2e-5 rms (<= ~1.5e-4 observed), which is why K3 re-checks in fp32 every row whose
// top-2 gap or distance to the threshold is <= delta.
//
// Decomposition (one CTA per SM, persistent over candidate tiles; template kCG = tcgen05 cta_group):
//   * candidates -> MMA M (TMEM lanes), references -> MMA N (TMEM columns).  A CTA keeps its 128-candidate
//     A tile (all of K) resident in shared memory and streams 256-reference B tiles, K-block by K-block,
//     out of L2 through a TMA/mbarrier ring: per 128 x 256 x K tile only B moves.
//   * kCG == 2 (default): two CTAs of a cluster (an SM pair) share every B tile -- each loads half of it and one
//     tcgen05.mma.cta_group::2 (M = 256) issued by the leader CTA reads A and B from both CTAs' shared memory
//     and writes 128 accumulator rows into each CTA's TMEM.
//   * warp 0: TMA producer, warp 1: tcgen05.mma issuer + TMEM owner -- one elected thread each, ring positions and
//     phases carried incrementally.  warps 2-9: epilogue, one thread per (candidate row, column half): the
//     max/argmax over references is a pure in-register reduction over TMEM columns -- no shuffles; the two column
//     halves of a row are merged through shared memory once per candidate tile.  kNorm: warps 10-11 L2-normalise
//     the fp32 rows of the CTA's next candidate tile (K1 inside K2) -- into the fp16 workspace, or (stage32, 128-d rows)
//     from TMA-staged fp32 rows straight into the swizzled A stage; in stage32 they also run the end-of-tile work
//     (merge of the column halves, classification, K3's lists) for the epilogue warps.
//   * the accumulator is double buffered in TMEM (2 x 256 of the 512 columns): the MMAs of reference tile
//     t+1 overlap the epilogue of tile t.
//   * epilogue per reference tile: four tcgen05.ld in flight -> stage released -> four 3-input-max trees -> the update
//     path update_grid (X/Y group maxima locate the single in-window column; group tests on the FMA pipe deliver the
//     groups' count and bit masks), unconditional for short reference sets, behind one branch on the tile maximum for
//     long ones.  Ascending column order + strict '>' = np.argmax first occurrence.  The running top-4 (+ the "hidden
//     column" state: the part with several in-window columns and its X/Y masks) is what K3 needs to make the index and
//     keep bit exact in fp32.  Duplicate reference rows may have been folded before (ffr_dedup.cu): columns then map back
//     to original indices through ref_map in the tail.
#include <cuda.h>
#include <stdlib.h>

#include <atomic>
#include <mutex>
#include <type_traits>

#include "ffr_common.cuh"

namespace ffr {

namespace {

constexpr int kTileM = 128;          // candidates per CTA tile (TMEM lanes)
constexpr int kTileN = 256;          // references per accumulator stage (TMEM columns), A-from-shared-memory variant
constexpr int kBlockK = 64;          // fp16 per 128-byte swizzle row
constexpr int kUmmaK = 16;
constexpr int kMaxAStages = 4;
constexpr int kMaxBStages = 16;
constexpr uint32_t kABlockBytes = kTileM * kBlockK * 2;      // 16 KiB: one K-block of the A tile
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kSmemLimit = 232448;                       // 227 KiB opt-in maximum
constexpr uint32_t kBarrierBytes = 1024;                      // mbarriers + TMEM slot
constexpr int kStageRows = 32;                                // stage32: fp32 candidate rows per staging buffer
constexpr uint32_t kStageBytes = kStageRows * 128 * 4;        // 16 KiB: 32 rows x 128 floats (dim_pad == 128 only)
constexpr int kMaxSBufs = 6;
constexpr uint32_t kMergeBytes = kTileM * 11 * 4;             // top-4 + hidden-column state hand-over of the other column half
// per kernel variant: extra = kBarrierBytes + (column parts - 1) * kMergeBytes

// running top-4 scores of one candidate (first three with their reference index): what K3 needs to decide in fp32
struct Top3 {
    float b1, b2, b3, b4;
    int32_t i1, i2, i3;
};

// Columns that were inside the window when they were seen but were NOT inserted one by one.  amb = the largest maximum of a
// 128-column part with several in-window columns (flag-only update path) and base = that part's first reference; amb2 = the
// largest such maximum of any OTHER part or 32-column chunk (exact path: further in-window columns of a chunk).  At the end
// of the candidate tile: amb2 still inside the window -> the whole reference set is rescanned in fp32 (K3b); only amb inside
// it -> K3 rescans just the 128 references of that part; neither -> nothing hidden matters any more.
struct Hidden {
    float amb, amb2;
    int32_t base;
    int32_t mask;       // of the part `base` names: bits 0-15 = X groups (columns 8a..8a+7), bits 16-23 = Y groups (column mod 8) that
                        // reached the window floor when the part was seen -- its in-window columns are among {8a + b}
};

// The two column halves of a candidate row merged (end of the candidate tile).  Their leading parts are joined into ONE span
// when they are ADJACENT (first columns 128 apart: the two halves of one reference tile, or the upper half of one and the
// lower half of the next) -- a group of near-identical references that straddles a part boundary puts several in-window columns
// into both, and without this every such row went to the full rescan.  xm: X-group bits of the span's first part in bits
// 0-15, of its second part (if any) in bits 16-31; ym: the union of their Y-group bits (a superset of the in-window columns).
struct HiddenM {
    float amb, amb2;
    int32_t base;       // first column of the span
    uint32_t xm, ym;
};

__device__ __forceinline__ HiddenM hidden_single(const Hidden& a) {
    HiddenM m;
    m.amb = a.amb; m.amb2 = a.amb2; m.base = a.base;
    m.xm = static_cast<uint32_t>(a.mask) & 0xFFFFu;
    m.ym = (static_cast<uint32_t>(a.mask) >> 16) & 0xFFu;
    return m;
}

__device__ __forceinline__ HiddenM hidden_merge(const Hidden& a, const Hidden& b) {
    constexpr int32_t kPart = kTileN / 2;
    const bool both = a.amb > -INFINITY && b.amb > -INFINITY;
    const bool a_first = a.base < b.base;
    const int32_t gap = a_first ? b.base - a.base : a.base - b.base;
    const uint32_t xa = static_cast<uint32_t>(a.mask) & 0xFFFFu, xb = static_cast<uint32_t>(b.mask) & 0xFFFFu;
    const uint32_t ya = (static_cast<uint32_t>(a.mask) >> 16) & 0xFFu, yb = (static_cast<uint32_t>(b.mask) >> 16) & 0xFFu;
    HiddenM m;
    if (both && gap == kPart) {                        // adjacent: one span of two parts, nothing "hidden elsewhere" added
        m.amb = fmaxf(a.amb, b.amb);
        m.amb2 = fmaxf(a.amb2, b.amb2);
        m.base = a_first ? a.base : b.base;
        m.xm = a_first ? (xa | (xb << 16)) : (xb | (xa << 16));
        m.ym = ya | yb;
    } else {                                           // the larger part maximum leads, the other is "a second part"
        const bool b_leads = b.amb > a.amb;
        m.amb = fmaxf(a.amb, b.amb);
        m.amb2 = fmax3(a.amb2, b.amb2, fminf(a.amb, b.amb));
        m.base = b_leads ? b.base : a.base;
        m.xm = b_leads ? xb : xa;
        m.ym = b_leads ? yb : ya;
    }
    return m;
}

__device__ __forceinline__ void top3_insert(Top3& t, float v, int32_t idx) {
    const bool g1 = v > t.b1, g2 = v > t.b2, g3 = v > t.b3, g4 = v > t.b4;
    t.b4 = g3 ? t.b3 : (g4 ? v : t.b4);
    t.i3 = g2 ? t.i2 : (g3 ? idx : t.i3);
    t.b3 = g2 ? t.b2 : (g3 ? v : t.b3);
    t.i2 = g1 ? t.i1 : (g2 ? idx : t.i2);
    t.b2 = g1 ? t.b1 : (g2 ? v : t.b2);
    t.i1 = g1 ? idx : t.i1;
    t.b1 = g1 ? v : t.b1;
}

// merge variant: the two column halves interleave in index order, so ties are broken by the smaller index
__device__ __forceinline__ void top3_merge_insert(Top3& t, float v, int32_t idx) {
    const bool g1 = (v > t.b1) || (v == t.b1 && idx < t.i1);
    const bool g2 = (v > t.b2) || (v == t.b2 && idx < t.i2);
    const bool g3 = (v > t.b3) || (v == t.b3 && idx < t.i3);
    const bool g4 = v > t.b4;
    t.b4 = g3 ? t.b3 : (g4 ? v : t.b4);
    t.i3 = g2 ? t.i2 : (g3 ? idx : t.i3);
    t.b3 = g2 ? t.b2 : (g3 ? v : t.b3);
    t.i2 = g1 ? t.i1 : (g2 ? idx : t.i2);
    t.b2 = g1 ? t.b1 : (g2 ? v : t.b2);
    t.i1 = g1 ? idx : t.i1;
    t.b1 = g1 ? v : t.b1;
}

// Update path of the epilogue.  v: 32 consecutive scores of this thread's candidate, cmax their maximum, base = reference
// index of v[0]; called only when cmax reaches gate = running best - delta.  After this chunk the window is
// [max(best, cmax) - delta, ...]; the chunk maximum is inserted at its first column (ascending columns + strict '>' in
// top3_insert = np.argmax first occurrence).  Nearly always it is the only column of the chunk inside the window; when
// it is not, the other columns are NOT inserted: the row remembers the largest such chunk maximum in `amb`, and if
// that is still inside the window of the final best (amb >= best - delta) the row goes to the full fp32 rescan (K3b),
// which sees every reference.  Hidden columns are <= their chunk maximum, so amb < best - delta proves they are
// irrelevant.  This keeps the path to ~110 instructions; the ordered insertion of every in-window column it
// replaces was ~600 and made the whole loop body too large for the instruction cache to stream.
__device__ __forceinline__ void update_chunk(const float (&v)[32], float cmax, int32_t base, float delta, Top3& t,
                                             float& gate, float& amb) {           // amb: Hidden::amb2 of the caller
    const float w = fmaxf(t.b1, cmax) - delta;
    uint32_t g[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {                      // independent chains (FSETP + SEL + 3-input add): 2.5 ops per column
        g[k] = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) g[k] |= (v[8 * k + j] >= w) ? (1u << (8 * k + j)) : 0u;
    }
    uint32_t ge = (g[0] | g[1]) | (g[2] | g[3]);
    if (ge & (ge - 1)) {                               // several columns inside the window (rare)
        amb = fmaxf(amb, cmax);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            g[k] = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) g[k] |= (v[8 * k + j] == cmax) ? (1u << (8 * k + j)) : 0u;
        }
        ge = (g[0] | g[1]) | (g[2] | g[3]);
    }
    if (ge != 0) top3_insert(t, cmax, base + __ffs(ge) - 1);      // (ge == 0 only with NaN scores: zero-norm rows)
    gate = t.b1 - delta;
}

// Batched form of the update path for SHORT reference sets, where nearly every chunk of every tile reaches the gate in
// some lane (a warp pays for the union of its lanes' record-setting chunks: with 1000 references that is all of them) and
// the sequential form is a chain of dependent ~110-instruction blocks at IPC 0.3.  All kC chunks of the part are masked
// against ONE floor w0 = max(best, part maximum) - delta: a column below w0 is outside the window once this part has been
// seen, so nothing that could matter later is skipped, and the kC mask builds are independent instruction streams.
template <int kC>
__device__ __forceinline__ void update_part(const float (&v)[kC][32], const float (&cm)[kC], float m, int32_t base0, float delta,
                                            Top3& t, float& gate, float& amb) {
    const float w0 = fmaxf(t.b1, m) - delta;
    uint32_t ge[kC];
#pragma unroll
    for (int c = 0; c < kC; ++c) {
        uint32_t g[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            g[k] = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) g[k] |= (v[c][8 * k + j] >= w0) ? (1u << (8 * k + j)) : 0u;
        }
        ge[c] = (g[0] | g[1]) | (g[2] | g[3]);
    }
#pragma unroll
    for (int c = 0; c < kC; ++c) {
        if (ge[c] != 0) {
            uint32_t pos = ge[c];
            if (pos & (pos - 1)) {                                // several columns of this chunk inside the window (rare)
                amb = fmaxf(amb, cm[c]);
                uint32_t g[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    g[k] = 0;
#pragma unroll
                    for (int j = 0; j < 8; ++j) g[k] |= (v[c][8 * k + j] == cm[c]) ? (1u << (8 * k + j)) : 0u;
                }
                pos = (g[0] | g[1]) | (g[2] | g[3]);
            }
            if (pos != 0) top3_insert(t, cm[c], base0 + c * 32 + __ffs(pos) - 1);
        }
    }
    gate = t.b1 - delta;
}

// maxima of the four 8-column groups of a chunk: the first level of the chunk's max tree (0.5 instruction per score)
__device__ __forceinline__ void group_max8(const float (&v)[32], float (&s)[4]) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
        s[k] = fmax3(fmax3(v[8 * k + 0], v[8 * k + 1], v[8 * k + 2]), fmax3(v[8 * k + 3], v[8 * k + 4], v[8 * k + 5]),
                     fmaxf(v[8 * k + 6], v[8 * k + 7]));
}

__device__ __forceinline__ float chunk_max(const float (&v)[32]) {
    float s[4];
    group_max8(v, s);
    return fmax3(s[0], s[1], fmaxf(s[2], s[3]));
}

// maximum of N registers as a tree of 3-input max
template <int N>
struct MaxTree {
    static __device__ __forceinline__ float run(const float (&a)[N]) {
        constexpr int M = (N + 2) / 3;
        float b[M];
#pragma unroll
        for (int i = 0; i < M; ++i) {
            if (3 * i + 2 < N)      b[i] = fmax3(a[3 * i], a[3 * i + 1], a[3 * i + 2]);
            else if (3 * i + 1 < N) b[i] = fmaxf(a[3 * i], a[3 * i + 1]);
            else                    b[i] = a[3 * i];
        }
        return MaxTree<M>::run(b);
    }
};
template <>
struct MaxTree<1> {
    static __device__ __forceinline__ float run(const float (&a)[1]) { return a[0]; }
};

// "Grid" form of the update path: straight-line, ~130 instructions per part whatever the data, instead of ~80 per chunk
// to build column masks.  The kC*32 columns of the part are seen as a (kC*4) x 8 grid: X group a = columns 8a..8a+7 (their
// maxima sx are the first level of the max tree the hot loop computes anyway), Y group b = the kC*4 columns with
// (column mod 8) == b.  A column >= w0 puts its X group AND its Y group at >= w0, and an X and a Y group share exactly one
// column -- so when exactly one X group and one Y group reach the floor there is exactly ONE column inside the window, it
// is column 8a + b, and its score is the part maximum m: insert it, done.  Only when two groups of either kind reach the
// floor (two columns of one part within delta of each other, or exact ties: rare) does the thread fall back to the exact
// per-column masks of update_part.  Same floor, same insertions: results are identical.
//
// The epilogue is bound by the ALU pipe (FMNMX / FSETP / SEL / IADD3 issue every other cycle per scheduler) while the FMA
// pipe idles, so the group tests run THERE: x = sat((s - w1) * 2^60) is 1.0 for s > w1 and 0.0 otherwise (one FFMA.SAT; w1
// = just below w0, so "> w1" holds for every s >= w0), and acc = sum x * (2^17 + 2^g) carries the number of groups at the floor
// and their bit mask (one FFMA per group, exact in fp32).  (The floor is at most an ulp-ish lower than w0: the window only
// gets wider, and the fall-back path uses w0 itself.)
template <int kC>
__device__ __forceinline__ void update_grid(const float (&v)[kC][32], const float (&sx)[kC][4], const float (&cm)[kC], float m,
                                            int32_t base0, float delta, bool exact, Top3& t, float& gate, Hidden& hid) {
    constexpr float kBig = 1152921504606846976.0f;     // 2^60
    const float w0 = fmaxf(t.b1, m) - delta;
    const float w1 = fmaf(fabsf(w0), -1.1920929e-7f, w0) - 1.0e-30f;
    const float cb = -w1 * kBig;
    // Each group test adds 2^17 + 2^g when group g reaches the floor: the (exact, < 2^22) sum carries the NUMBER of such groups in
    // bits 17.. and their BIT MASK below -- the single in-window column of the common case is decoded from the two masks, and
    // with several (flag-only path) the masks tell K3 which of the part's 128 references it has to look at.
    static_assert(kC * 4 <= 16, "X-group mask is 16 bits");
    constexpr float kCnt = 131072.0f;                   // 2^17
    float ax[2] = {0.f, 0.f}, ay[2] = {0.f, 0.f};
#pragma unroll
    for (int c = 0; c < kC; ++c)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int g = c * 4 + k;
            ax[g & 1] = fmaf(__saturatef(fmaf(sx[c][k], kBig, cb)), kCnt + static_cast<float>(1 << g), ax[g & 1]);
        }
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        float col[kC * 4];
#pragma unroll
        for (int c = 0; c < kC; ++c)
#pragma unroll
            for (int k = 0; k < 4; ++k) col[c * 4 + k] = v[c][8 * k + b];
        ay[b & 1] = fmaf(__saturatef(fmaf(MaxTree<kC * 4>::run(col), kBig, cb)), kCnt + static_cast<float>(1 << b), ay[b & 1]);
    }
    // (NaN scores of a zero-norm row: sat(NaN) = 0 on this path, the sums stay 0 -> "below the window")
    const int32_t ix = __float2int_rn(ax[0] + ax[1]), iy = __float2int_rn(ay[0] + ay[1]);
    const int32_t nx = ix >> 17, ny = iy >> 17;
    const int32_t mx = ix & 0x1FFFF, my = iy & 0x1FFFF;
    const bool multi = max(nx, ny) >= 2;               // several columns of this part inside the window (rare per thread)
    if (exact && multi) {
        // (a fall-back at 8-column granularity -- one divergent region per X group at the floor -- gave fewer full rescans
        // but was slower than the per-chunk masks: 16 reconvergence regions in the loop body cost more than they save)
        update_part<kC>(v, cm, m, base0, delta, t, gate, hid.amb2);
        return;
    }
    // !exact: no second path at all.  "Rare per thread" is not rare per accumulator stage -- the MMA waits for the slowest
    // of the 16 warps of a CTA pair, and with ~0.3 % of (row, part) pairs taking a 400-instruction detour most tiles had one.
    // Instead the part maximum goes in with a placeholder column (the part's first) and the row remembers the part: if its
    // maximum is still within delta of the final best, K3 rescans the 128 references of THAT part in fp32 (plus the row's
    // other tracked candidates) -- or every reference, if a second such part is inside the window too; if it is not, nothing
    // of this part matters any more.
    // (sums < 1: the part is below the window, or NaN scores of a zero-norm row -- inserting -inf is a no-op)
    const float ins = min(nx, ny) >= 1 ? m : -INFINITY;
    const int32_t col = multi ? 0 : 8 * (31 - __clz(mx | 1)) + (31 - __clz(my | 1));                   // 8 a + b
    const bool lead = multi && m > hid.amb;
    hid.amb2 = multi ? fmaxf(hid.amb2, fminf(hid.amb, m)) : hid.amb2;
    hid.amb = lead ? m : hid.amb;
    hid.base = lead ? base0 : hid.base;
    hid.mask = lead ? (mx | (my << 16)) : hid.mask;
    top3_insert(t, ins, base0 + col);
    gate = t.b1 - delta;
}

__device__ __forceinline__ void mask_chunk(float (&v)[32], int valid) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = (j < valid) ? v[j] : -INFINITY;
}

// ---- cluster / cta_group::2 PTX -------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;     // shared::cluster address of the same offset in the pair's CTA 0
// Arrive on CTA 0's copy of a barrier WITHOUT release semantics: for "this warp has finished READING the accumulator stage"
// (t_empty).  The reads are complete (tcgen05.wait::ld) and ordered by tcgen05.fence::before_thread_sync; no generic-proxy
// writes need to become visible.  The .release.cluster form compiles to MEMBAR.ALL.GPU + arrive, ~1 us per reference tile.
__device__ __forceinline__ void mbar_arrive_leader_relaxed(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, 0;\n\t"
        "mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(smem_u32(bar)) : "memory");
}
// Default semantics (.release at CTA scope) on the leader's barrier: what a producer warp needs after fence.proxy.async when
// the data it wrote is only ever read through the async proxy (the leader's tcgen05.mma reading THIS CTA's shared memory).
// The .release.cluster form above costs a MEMBAR.ALL.GPU (~1 us) per arrive.
__device__ __forceinline__ void mbar_arrive_leader_cta(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, 0;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_2d_cg2(void* smem_dst, const void* desc, uint64_t* bar, int32_t c0, int32_t c1,
                                                uint64_t cache_hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(desc), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "l"(cache_hint)
        : "memory");
}
__device__ __forceinline__ void umma_f16_cg2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_cg2(uint64_t* bar) {         // arrives on the barrier in BOTH CTAs
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(smem_u32(bar)), "h"(static_cast<uint16_t>(3)) : "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* smem_dst) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(smem_dst)), "n"(kCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t n) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t n) {
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory");
}

__device__ __forceinline__ void mbar_wait_timed(uint64_t* bar, uint32_t parity, bool on, unsigned long long& acc) {
    if (!on) { mbar_wait(bar, parity); return; }
    const long long t0 = clock64();
    mbar_wait(bar, parity);
    acc += static_cast<unsigned long long>(clock64() - t0);
}

// wait with cluster-scope acquire: the arrivals come from the PEER CTA's normaliser warps (stage32), whose generic-proxy
// shared-memory writes the leader's MMAs are about to read
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (ok == 0);
}

struct KParams {
    int64_t n_ref, n_cand;          // n_ref: rows of the fp16 reference matrix the tensor map describes
    const int32_t* n_ref_dev;      // duplicate references folded (ffr_dedup.cu): the number of UNIQUE rows, known on the device only;
    const int32_t* ref_map;        // ... rows [*n_ref_dev, n_ref) are stale, and column i stands for original reference ref_map[i]
    int32_t kb_count, a_stages, b_stages;
    float thr, delta, thr_band;
    int64_t ref_index_base;
    uint8_t* keep;
    int32_t* best_idx;
    float* best_val;
    RecheckLists lists;
    int no_recheck;
    float band_tol;                // no_recheck only: rows with |best - thr| <= band_tol are listed by the tail (with the re-check K3 lists them)
    int32_t* band_count;
    int64_t* band_rows;
    int64_t band_cap;
    float* dbg_scores;
    const float* cand32;           // kNorm: original fp32 candidate rows [n_cand, dim]
    __half* cand16;                // kNorm: where the normalised fp16 rows go (leading dimension kb_count * 64)
    int32_t dim;                   // kNorm: true embedding size (row pitch of cand32)
    int grid_updates;              // epilogue: unconditional grid update path (n_ref <= FFR_GRID_UPDATE_REFS, default 8192)
    int grid_exact;                // update_grid: a part with several in-window columns takes the exact per-column path (1) or only
                                   // flags the row for the full fp32 rescan (0: branch-free; default for dim <= 256, FFR_GRID_EXACT)
    int stage32;                   // kNorm, dim_pad == 128: fp32 candidate rows are staged through shared memory by TMA and the normaliser
                                   // warps write the swizzled fp16 A tile directly (no global scratch, no K1 pass at ANY n_ref)
    int s_bufs;                    // stage32: staging ring depth (buffers of kStageRows rows)
    unsigned long long* prof;      // optional [gridDim.x][32] stall-cycle counters (diagnostics)
    // kEuclid: score = acc + ref_bias[col] * cand_scale[row] (DESIGN.md section 4, "Euclid on the tensor cores")
    const float* ref_bias;         // -|r|^2 * 2^-f / 2 per (compact) reference column, zero padded to a multiple of kTileN
    const float* cand_scale;       // 1 / |c| per candidate row (K1)
    const float* bias_max;         // max |ref_bias| (device scalar): sizes the per-row window
    // kSelf: the candidates are rows [self_row0, self_row0 + n_cand) of the reference matrix (DESIGN.md section 4, "Self mode")
    int64_t self_row0;
    int self_mode;                 // FFR_SELF_OTHERS | FFR_SELF_EARLIER
};

// End of a candidate tile, once per row (the two column halves merged): classify_row writes keep / index / score and decides
// which of K3's lists the row goes to; append_rows adds the rows of a warp (kNR per lane) to the lists, warp-aggregated, with
// at most ONE atomic per list and all of them in flight together (a returning global atomic is ~700 cycles: one per list and
// row, one after the other, was most of the tail's time).  The whole warp must call append_rows together.
//   1 pair : near-tie / near-threshold row with at most three candidates       -> pair record (front of `recs`)
//   2 part : un-inserted in-window columns confined to ONE 128-reference part   -> part record (back of `recs`)
//   3 full : a fourth score or hidden columns of a second part inside the window -> full rescan list
struct RowOut {
    int cls;
    RecheckRec rec;
};

// kEuclid: the row's window is delta_e (not p.delta), and force_full sends the row to the full rescan whatever its scores.
// kSelf: `none` = the row has no eligible reference (row 0 in FFR_SELF_EARLIER): index -1, score -inf, no re-check, no band.
template <bool kEuclid = false, bool kSelf = false>
__device__ __forceinline__ RowOut classify_row(const KParams& p, const Top3& t, const HiddenM& hid, int64_t row,
                                               float delta_e = 0.f, bool force_full = false, bool none = false) {
    RowOut o;
    if constexpr (kSelf) {
        if (none) {
            if (row < p.n_cand) {
                p.keep[row] = 0;
                p.best_idx[row] = -1;
                if (p.best_val != nullptr) p.best_val[row] = -INFINITY;
            }
            o.cls = 0;
            o.rec.row = static_cast<int32_t>(row);
            o.rec.idx1 = o.rec.idx2 = o.rec.idx3 = -1;
            return o;
        }
    }
    const auto delta = [&]() { return kEuclid ? delta_e : p.delta; };
    const bool valid = row < p.n_cand;
    const bool near_tie = (t.i2 >= 0) && (t.b1 - t.b2 <= delta());
    const bool near_thr = fabsf(t.b1 - p.thr) <= p.thr_band;
    // un-inserted columns may be inside the window: of ONE part (K3 rescans its 128 references), or of more
    const bool hid2 = hid.amb2 > -INFINITY && hid.amb2 >= t.b1 - delta();
    const bool hid1 = hid.amb > -INFINITY && hid.amb >= t.b1 - delta();
    const bool forced = kEuclid && force_full;
    const bool flagged = valid && !p.no_recheck && (forced || near_tie || near_thr || hid1 || hid2);
    const bool full = flagged && (forced || hid2 || t.b1 - t.b4 <= delta());   // four or more inside the window, or hidden ones anywhere
    const bool part = flagged && !full && hid1;                        // hidden columns in one known part
    const int32_t* map = p.ref_map;                                     // duplicate references folded: compact -> original index
    const auto orig = [&](int32_t i) { return (map != nullptr && i >= 0) ? map[i] : i; };
    if (valid) {
        p.keep[row] = (t.b1 >= p.thr) ? 1 : 0;
        p.best_idx[row] = static_cast<int32_t>(orig(t.i1) + p.ref_index_base);
        if (p.best_val != nullptr) p.best_val[row] = t.b1;
        if (p.band_count != nullptr && fabsf(t.b1 - p.thr) <= p.band_tol) {     // (no re-check: fp16-operand score)
            const int32_t slot = atomicAdd(p.band_count, 1);
            if (p.band_rows != nullptr && slot < p.band_cap) p.band_rows[slot] = row;
        }
    }
    o.cls = !flagged ? 0 : (full ? 3 : (part ? 2 : 1));
    o.rec.row = static_cast<int32_t>(row);
    o.rec.idx1 = o.rec.idx2 = o.rec.idx3 = -1;
    if (o.cls == 2) {
        // The part's own placeholder entry (and anything else inside the part) is covered by K3's scan of the part.  The record
        // names the span (one part or two adjacent ones) by its first COMPACT column and carries the X / Y group masks (the
        // in-window columns are among {8a + b}) plus ONE tracked candidate outside the span, by original index; a second one
        // makes it a full rescan.  (Layout: ffr_recheck.cu, K3p.)
        const int32_t span = (hid.xm >> 16) != 0u ? kTileN : kTileN / 2;     // one part, or two adjacent ones
        const auto outside = [&](float b, int32_t i) {
            return i >= 0 && b >= t.b1 - delta() && (i < hid.base || i >= hid.base + span);
        };
        int32_t e = -1;
        int ne = 0;
        if (outside(t.b1, t.i1)) { e = t.i1; ++ne; }
        if (outside(t.b2, t.i2)) { e = ne ? e : t.i2; ++ne; }
        if (outside(t.b3, t.i3)) { e = ne ? e : t.i3; ++ne; }
        if (ne > 1) o.cls = 3;
        o.rec.idx1 = static_cast<int32_t>(static_cast<uint32_t>(hid.base >> 7) | (hid.ym << 24));   // (base: a multiple of 128, < 2^31)
        o.rec.idx2 = orig(e);
        o.rec.idx3 = static_cast<int32_t>(hid.xm);
    } else if (o.cls == 1) {
        o.rec.idx1 = orig(t.i1);
        o.rec.idx2 = near_tie ? orig(t.i2) : -1;
        o.rec.idx3 = (near_tie && t.i3 >= 0 && t.b1 - t.b3 <= delta()) ? orig(t.i3) : -1;
    }
    return o;
}

template <int kNR>
__device__ __forceinline__ void append_rows(const KParams& p, const RowOut (&o)[kNR], int lane) {
    uint32_t m[3][kNR];
    int tot[3] = {0, 0, 0};
#pragma unroll
    for (int k = 0; k < kNR; ++k)
#pragma unroll
        for (int l = 0; l < 3; ++l) {
            m[l][k] = __ballot_sync(0xffffffffu, o[k].cls == l + 1);
            tot[l] += __popc(m[l][k]);
        }
    if ((tot[0] | tot[1] | tot[2]) == 0) return;
    int32_t base[3] = {0, 0, 0};
    if (lane == 0) {                                   // the (up to three) atomics go out back to back
        if (tot[0] != 0) base[0] = atomicAdd(&p.lists.hdr->recheck_count, tot[0]);
        if (tot[1] != 0) base[1] = atomicAdd(&p.lists.hdr->part_count, tot[1]);
        if (tot[2] != 0) base[2] = atomicAdd(&p.lists.hdr->full_count, tot[2]);
    }
#pragma unroll
    for (int l = 0; l < 3; ++l) base[l] = __shfl_sync(0xffffffffu, base[l], 0);
    const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
    for (int k = 0; k < kNR; ++k) {
        if (o[k].cls == 1) {                           // pair records grow UP from the front of the record array ...
            const int64_t slot = base[0] + __popc(m[0][k] & lt);
            if (slot < p.lists.rec_cap) p.lists.recs[slot] = o[k].rec;
        } else if (o[k].cls == 2) {                    // ... part records DOWN from its end: a row is in exactly one list
            const int64_t slot = p.lists.rec_cap - 1 - (base[1] + __popc(m[1][k] & lt));
            if (slot >= 0) p.lists.recs[slot] = o[k].rec;
        } else if (o[k].cls == 3) {
            const int64_t slot = base[2] + __popc(m[2][k] & lt);
            if (slot < p.lists.full_cap) {
                p.lists.full_rows[slot] = o[k].rec.row;
                p.lists.full_keys[slot] = 0ull;
                if (slot % kFullGroup == 0) p.lists.full_ctr[slot / kFullGroup] = 0;
            }
        }
#pragma unroll
        for (int l = 0; l < 3; ++l) base[l] += __popc(m[l][k]);
    }
}

// Self mode, FFR_SELF_EARLIER: candidate tile t only needs the reference tiles up to the last one with a column below its last
// row.  The TMA producer, the MMA thread and the epilogue derive the same range from the tile index.  (Candidate tiles stay
// dealt round-robin: with per-tile work growing linearly, a reversed order gives the busiest CTA pair the same sum -- the
// last-wave imbalance is the wave quantisation the gallery call has too; tools/bench_self.py prints it.)
__device__ __forceinline__ int32_t self_rt_end(const KParams& p, int64_t ct, int32_t n_rt) {
    if (p.self_mode != FFR_SELF_EARLIER) return n_rt;
    constexpr int64_t kPair = 2 * kTileM;                              // (self mode runs cta_group::2)
    const int64_t last = ct * kPair + (kPair - 1) < p.n_cand ? ct * kPair + (kPair - 1) : p.n_cand - 1;
    return static_cast<int32_t>((p.self_row0 + last + kTileN - 1) / kTileN);
}

// kCG: tcgen05 cta_group (1|2).  Eight epilogue warps = 4 TMEM lane quadrants x 2 column halves.
// kNormMode != 0 (kNorm): K1 for the candidates runs INSIDE this kernel.  Two extra "normaliser" warps (the hardware allocates warps in
// fours, so 10 warps cost 12 anyway) read the fp32 rows of the CTA's NEXT candidate tile, L2-normalise them exactly like K1
// and write the fp16 rows into the workspace, while the tensor core works on the current tile; the TMA producer waits
// for a per-CTA counter before it loads a tile.  The rows come back through L2, HBM sees the fp32 embeddings once, and
// the 0.6 ms K1 pass over 1.25 M x 512 disappears behind the MMAs (the kernel needs < 10 % of K1's bandwidth).
// kExact / kAlways: the two epilogue policies as COMPILE-TIME constants (0 | 1; 2 = read the run-time flag, used by the
// instrumented build and cta_group::1).  kExact = 0 removes the ~1100-instruction exact fall-back (update_part) from the
// hot loop's body altogether; kAlways picks the unconditional or the gated update path.
// kEuclid: the Euclid decision rule (K1 schedule, cta_group::2, production policies only): every score gets the per-reference
// bias scaled by the row's 1 / |c| before the max trees, and the row's window widens with that bias (DESIGN.md section 4).
// kSelf: self mode (ffr_filter_self; K1 schedule, cta_group::2, production policies only).  A reference tile that holds a
// column the row may not match -- its own (FFR_SELF_OTHERS) or any at or after it (FFR_SELF_EARLIER) -- runs the masked copy of
// the epilogue body; FFR_SELF_EARLIER stops every role at the last reference tile with a column below the candidate tile's last
// row.
template <int kCG, int kNormMode, int kExact, int kAlways, bool kInstr, bool kEuclid = false, bool kSelf = false>
__global__ void __launch_bounds__(64 + 32 * 8 + (kNormMode ? 64 : 0), 1)   // 10 warps are allocated as 12: <= 168 registers
filter_mma_kernel(const __grid_constant__ CUtensorMap tmap_cand, const __grid_constant__ CUtensorMap tmap_ref,
                  const __grid_constant__ CUtensorMap tmap_cand32, const KParams p) {
    // kNormMode: 0 = the candidates' fp16 rows come from K1, 1 = normaliser warps with global loads + fp16 scratch, 2 = stage32.
    // (Separate instantiations: with stage32 as a run-time branch its mere presence cost the dim-512 kernel 1.5 % of wall clock.)
    // kInstr: the instrumented build (in-kernel cycle counters, score dump).  The production
    // instantiation contains none of it: the counters alone were half a dozen spilled 64-bit values per role.
    static_assert(!kSelf || (kCG == 2 && kNormMode == 0 && !kInstr), "self mode runs on the K1 schedule, cta_group::2, production build");
    constexpr bool kNorm = kNormMode != 0;
    constexpr bool st32 = kNormMode >= 2;
    // stage32 comes in two forms: kNormMode 2 hands the end-of-tile work (merge of the column halves, classification, K3's
    // lists) to the two normaliser warps -- right when the epilogue paces the kernel (>= 2 reference tiles per candidate tile);
    // kNormMode 3 keeps it in the epilogue warps -- right when there is ONE reference tile per candidate tile (<= 256
    // references: the HBM-bound regime), where the normaliser warps are the busy ones and the epilogue has cycles to spare.
    constexpr bool kOffload = kNormMode == 2;
    constexpr int kEW = 8;                                          // epilogue warps
    constexpr int kAccN = kTileN;                                   // references per accumulator stage
    const unsigned long long* const prof_on = kInstr ? p.prof : nullptr;
    constexpr int kParts = kEW / 4;                                 // column parts per reference tile
    constexpr int kChunksPerPart = (kAccN / 32) / kParts;
    constexpr uint32_t kBRows = kAccN / kCG;                        // B rows this CTA loads per K-block
    constexpr uint32_t kBStageBytes = kBRows * kBlockK * 2;         // 32 KiB (kCG 1) / 16 KiB (kCG 2)
    extern __shared__ __align__(1024) uint8_t smem[];               // SWIZZLE_128B atoms need 1024-byte alignment
    const uint32_t a_stage_bytes = static_cast<uint32_t>(p.kb_count) * kABlockBytes;
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem_a + static_cast<size_t>(p.a_stages) * a_stage_bytes;
    uint8_t* smem_s = smem_b + static_cast<size_t>(p.b_stages) * kBStageBytes;          // stage32: fp32 staging ring
    uint8_t* extra = smem_s + (st32 ? static_cast<size_t>(p.s_bufs) * kStageBytes : 0);
    uint64_t* a_full = reinterpret_cast<uint64_t*>(extra);
    uint64_t* a_empty = a_full + kMaxAStages;
    uint64_t* b_full = a_empty + kMaxAStages;
    uint64_t* b_empty = b_full + kMaxBStages;
    uint64_t* t_full = b_empty + kMaxBStages;
    uint64_t* t_empty = t_full + 2;
    uint64_t* s_full = t_empty + 2;
    uint64_t* s_empty = s_full + kMaxSBufs;
    uint64_t* m_full = s_empty + kMaxSBufs;                          // stage32: both column halves of a candidate tile have parked their state
    uint64_t* m_empty = m_full + 2;                                  // stage32: ... and the helper warps have merged + emitted it
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(m_empty + 2);
    uint32_t* norm_count = tmem_slot + 1;                            // kNorm: [2] candidate tiles finished by each normaliser warp
    uint32_t* cons_count = tmem_slot + 3;                            // kNorm: candidate tiles whose A loads have been issued
    float* merge = reinterpret_cast<float*>(extra + kBarrierBytes);  // [10][kTileM]; stage32: [2 slots][2 halves][10][kTileM]

    unsigned long long ts_entry = 0;
    if (prof_on != nullptr && threadIdx.x == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts_entry));
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t cta_rank = (kCG == 2) ? cluster_ctarank() : 0u;
    const bool leader = cta_rank == 0;
    const int64_t n_tiles = (p.n_cand + kTileM * kCG - 1) / (kTileM * kCG);   // tiles of the CTA pair
    const int64_t tile0 = blockIdx.x / kCG, tile_stride = gridDim.x / kCG;
    // duplicate references folded: the live row count is a device-side value written by the dedup kernels, which precede this
    // launch in plain stream order (the kernel is then NOT launched as K1's programmatic dependent)
    const int64_t n_ref = p.n_ref_dev != nullptr ? static_cast<int64_t>(__ldg(p.n_ref_dev)) : p.n_ref;
    const int32_t n_rt = static_cast<int32_t>((n_ref + kAccN - 1) / kAccN);

    if (threadIdx.x == 0) {
        if ((smem_u32(smem) & 1023u) != 0) __trap();
        tma_prefetch_desc(&tmap_cand);
        tma_prefetch_desc(&tmap_ref);
        if (st32) tma_prefetch_desc(&tmap_cand32);
        // stage32: A tiles are completed by the normaliser warps of BOTH CTAs (one arrive per warp) instead of TMA bytes
        for (int i = 0; i < kMaxAStages; ++i) { mbar_init(&a_full[i], st32 ? 2 * kCG : 1); mbar_init(&a_empty[i], 1); }
        for (int i = 0; i < kMaxSBufs; ++i) { mbar_init(&s_full[i], 1); mbar_init(&s_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&m_full[i], kEW); mbar_init(&m_empty[i], 2); }
        norm_count[0] = 0; norm_count[1] = 0; *cons_count = 0;
        for (int i = 0; i < kMaxBStages; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], kEW * kCG); }
        fence_barrier_init();
    }
    if (warp == 1) {
        if (kCG == 2) tmem_alloc_cg2<kTmemCols>(tmem_slot);
        else          tmem_alloc<kTmemCols>(tmem_slot);
    }
    tc_fence_before();
    if (kCG == 2) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (prof_on != nullptr && threadIdx.x == 0) {
        unsigned long long ts;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts));
        p.prof[blockIdx.x * 32 + 12] = ts - ts_entry;                  // ns: entry -> setup done (barriers, TMEM, cluster sync)
        p.prof[blockIdx.x * 32 + 15] = ts_entry;
    }

    if (warp == 0) {
        // ===================== TMA producer: ONE elected thread runs the whole loop =====================
        // (Inside `if (elect_one())` ptxas knows a single lane is active and emits plain UTMALDG / UTCHMMA; under
        // `if (lane == 0)` it wrapped each of them in a serialising vote loop, ~200 cycles per instruction.)  Ring
        // positions and phases are carried incrementally: a runtime `% stages` per K-block is a 25-instruction
        // division with MUFU latency on the critical path of every stage.
        if (elect_one()) {
            const bool pr = prof_on != nullptr;
            unsigned long long w_aempty = 0, w_bempty = 0;
            const long long t_begin = clock64();
            uint32_t as = 0, aph = 0, bs = 0, bph = 0, a_it = 0;
            // Programmatic dependent launch: this kernel may have started while K1 (fp16 references, and the candidates' fp16
            // rows when K1 normalises them) is still running.  stage32 reads the ORIGINAL fp32 candidates, which K1 never
            // touches: those loads go out first and only the first reference-tile load waits for K1.
            bool k1_done = false;
            if (!st32) { pdl_wait(); k1_done = true; }
            // stage32: the candidates arrive as fp32 rows in a ring of kStageRows-row staging buffers (four per tile); the
            // loads run as far ahead as the ring allows, independent of the A stages (the normaliser warps wait for those)
            const int64_t my_tiles = tile0 < n_tiles ? (n_tiles - tile0 + tile_stride - 1) / tile_stride : 0;
            const int64_t s_total = st32 ? my_tiles * (kTileM / kStageRows) : 0;
            int64_t s_next = 0;
            uint32_t sb = 0, sph = 0;
            auto try_issue_s = [&]() {
                while (s_next < s_total) {
                    if (!mbar_test_wait(&s_empty[sb], sph ^ 1)) return;
                    const int64_t t = tile0 + (s_next / (kTileM / kStageRows)) * tile_stride;
                    int32_t r0 = static_cast<int32_t>(t * (kTileM * kCG) + cta_rank * kTileM) +
                                 static_cast<int32_t>(s_next % (kTileM / kStageRows)) * kStageRows;
                    // No TMA box may lie ENTIRELY outside its tensor (see the B loads below: such boxes were measured to cost several
                    // times a normal tile, and crashed one configuration).  Rows past the last candidate are never emitted and the
                    // normaliser zeroes them (inv = 0): the last in-bounds rows are loaded in their place.  A column group that starts
                    // at or past `dim` (rows of 68..96 floats) is not loaded at all: the normaliser warps zeroed it once, and nothing
                    // overwrites it.
                    if (r0 >= p.n_cand) r0 = p.n_cand > kStageRows ? static_cast<int32_t>(p.n_cand) - kStageRows : 0;
                    const int n_groups = (p.dim + 31) >> 5;   // live 32-float column groups (3 or 4: dim_pad == 128)
                    mbar_expect_tx(&s_full[sb], (kStageBytes / 4) * n_groups);
#pragma unroll
                    for (int g = 0; g < 4; ++g)               // four 32-float (128-byte, swizzled) column groups of the rows
                        if (g < n_groups)
                            tma_load_2d(smem_s + sb * kStageBytes + g * (kStageBytes / 4), &tmap_cand32, &s_full[sb], g * 32, r0, kEvictFirst);
                    ++s_next;
                    if (++sb == static_cast<uint32_t>(p.s_bufs)) { sb = 0; sph ^= 1; }
                }
            };
            for (int64_t tile = tile0; tile < n_tiles; tile += tile_stride) {
                int32_t row0 = static_cast<int32_t>(tile * (kTileM * kCG) + cta_rank * kTileM);
                // (a fully out-of-bounds A box -- the peer CTA's half of a ragged last tile -- is replaced by the last in-bounds
                // rows: rows >= n_cand are never emitted)
                if (row0 >= p.n_cand) row0 = p.n_cand > kTileM ? static_cast<int32_t>(p.n_cand) - kTileM : 0;
                // The B stream does not depend on the candidate tile: it keeps flowing across tile boundaries, and this
                // tile's A loads go out the moment their stage is free (and, kNorm, the fp16 rows are written) -- probed
                // without blocking while the thread waits for B slots.  (Handing A back K-block by K-block during the last
                // reference tile removed the a_full wait in the in-kernel cycle counts -- 4308 -> 4180 per tile at dim 512 --
                // but the same-box wall clock of cfg3 got 4 % WORSE, 9.10 -> 9.46 ms: whole stages again.)
                bool need_a = true;
                if (st32) need_a = s_next < s_total;
                auto try_issue_a = [&]() {
                    if (st32) { try_issue_s(); need_a = s_next < s_total; return; }
                    if (kNorm && (ld_acquire_shared(&norm_count[0]) <= a_it || ld_acquire_shared(&norm_count[1]) <= a_it)) return;
                    if (!mbar_test_wait(&a_empty[as], aph ^ 1)) return;
                    if (leader) mbar_expect_tx(&a_full[as], a_stage_bytes * kCG);    // both CTAs' bytes land on the leader's barrier
                    for (int kb = 0; kb < p.kb_count; ++kb) {
                        uint8_t* dst = smem_a + as * a_stage_bytes + kb * kABlockBytes;
                        if (kCG == 2) tma_load_2d_cg2(dst, &tmap_cand, &a_full[as], kb * kBlockK, row0, kEvictFirst);
                        else          tma_load_2d(dst, &tmap_cand, &a_full[as], kb * kBlockK, row0, kEvictFirst);
                    }
                    if (kNorm) red_release_shared_add(cons_count, 1u);
                    need_a = false;
                };
                try_issue_a();
                if (!k1_done) { pdl_wait(); k1_done = true; }
                for (int rt = 0; rt < (kSelf ? self_rt_end(p, tile, n_rt) : n_rt); ++rt) {
                    int32_t rrow0 = rt * kAccN + static_cast<int32_t>(cta_rank * kBRows);
                    // A box that lies ENTIRELY past the last reference (the peer CTA's half of a last tile with <= 128 live
                    // references) is not loaded as such: measured, a tile with such a box costs 4-5 x a normal one (the MMA
                    // thread waits for b_full ~60 % of its time; cta_group::1, whose box is only partly out of bounds, and 129
                    // references do not show it).  Its columns are >= n_ref, i.e. masked to -inf by index whatever they hold,
                    // so the last in-bounds rows are loaded in its place.
                    if (kCG == 2 && rrow0 >= n_ref) rrow0 = n_ref > static_cast<int64_t>(kBRows) ? static_cast<int32_t>(n_ref) - static_cast<int32_t>(kBRows) : 0;
                    for (int kb = 0; kb < p.kb_count; ++kb) {
                        if (need_a) {
                            const long long tw0 = pr ? clock64() : 0;
                            while (!mbar_test_wait(&b_empty[bs], bph ^ 1)) { if (need_a) try_issue_a(); }
                            if (pr) w_bempty += static_cast<unsigned long long>(clock64() - tw0);
                        } else {
                            mbar_wait_timed(&b_empty[bs], bph ^ 1, pr, w_bempty);
                        }
                        if (leader) mbar_expect_tx(&b_full[bs], kBStageBytes * kCG);
                        uint8_t* dst = smem_b + bs * kBStageBytes;
                        if (kCG == 2) tma_load_2d_cg2(dst, &tmap_ref, &b_full[bs], kb * kBlockK, rrow0, kEvictLast);
                        else          tma_load_2d(dst, &tmap_ref, &b_full[bs], kb * kBlockK, rrow0, kEvictLast);
                        if (++bs == static_cast<uint32_t>(p.b_stages)) { bs = 0; bph ^= 1; }
                    }
                }
                if (need_a && !st32) {                      // fewer B loads than ring slots: nothing made the thread wait
                    const long long tw0 = pr ? clock64() : 0;
                    while (need_a) try_issue_a();
                    if (pr) w_aempty += static_cast<unsigned long long>(clock64() - tw0);
                }
                ++a_it;
                if (++as == static_cast<uint32_t>(p.a_stages)) { as = 0; aph ^= 1; }
            }
            while (s_next < s_total) try_issue_s();          // stage32: the last tiles' rows (every B load is out by now)
            if (pr) {
                p.prof[blockIdx.x * 32 + 0] = static_cast<unsigned long long>(clock64() - t_begin);
                p.prof[blockIdx.x * 32 + 1] = w_aempty;
                p.prof[blockIdx.x * 32 + 2] = w_bempty;
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== MMA issuer: one elected thread of the leader CTA =====================
        if (leader && elect_one()) {
            const bool pr = prof_on != nullptr;
            unsigned long long w_afull = 0, w_tempty = 0, w_bfull = 0;
            const long long t_begin = clock64();
            // UMMA smem descriptor, K-major SWIZZLE_128B: hi word is constant (SBO 1024 B, version 1, layout 2);
            // lo word = (address >> 4) | LBO(1) << 16, advanced by 2 (32 bytes) per K = 16 step.
            constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
            constexpr uint64_t kDescHi64 = static_cast<uint64_t>(kDescHi) << 32;
            constexpr int kSteps = kBlockK / kUmmaK;                        // MMAs per K-block
            const uint32_t b_lo_base = ((smem_u32(smem_b) & 0x3FFFFu) >> 4) | (1u << 16);
            const uint32_t idesc_full = umma_idesc_f16(kTileM * kCG, kAccN);
            uint32_t as = 0, aph = 0, bs = 0, bph = 0, acc = 0, tph = 0, t_it = 0;
            for (int64_t tile = tile0; tile < n_tiles; tile += tile_stride) {
                if (st32) {
                    const long long tw0 = pr ? clock64() : 0;
                    mbar_wait_cluster(&a_full[as], aph);
                    if (pr) w_afull += static_cast<unsigned long long>(clock64() - tw0);
                } else {
                    mbar_wait_timed(&a_full[as], aph, pr, w_afull);
                }
                tc_fence_after();
                const uint32_t a_lo0 = ((smem_u32(smem_a + as * a_stage_bytes) & 0x3FFFFu) >> 4) | (1u << 16);
                for (int rt = 0; rt < (kSelf ? self_rt_end(p, tile, n_rt) : n_rt); ++rt) {
                    mbar_wait_timed(&t_empty[acc], tph ^ 1, pr, w_tempty);
                    tc_fence_after();
                    uint32_t idesc = idesc_full;
                    if (kCG == 1) {                             // tail reference tile: only as many columns as needed
                        // (the cta_group::2 analogue -- N = 2 * ceil16(live) when the live references sit in CTA 0's half --
                        // is correct but did not pay: an N = 32 MMA costs ~100 cycles, and the same-box wall clock got worse)
                        const int64_t ncols = n_ref - static_cast<int64_t>(rt) * kAccN;
                        if (ncols < kAccN) idesc = umma_idesc_f16(kTileM * kCG, static_cast<uint32_t>((ncols + 15) & ~int64_t(15)));
                    }
                    const uint32_t d_tmem = tmem_base + acc * kAccN;
                    for (int kb = 0; kb < p.kb_count; ++kb) {
                        mbar_wait_timed(&b_full[bs], bph, pr, w_bfull);
                        tc_fence_after();
                        const uint32_t b_lo = b_lo_base + bs * (kBStageBytes >> 4);
#pragma unroll
                        for (int k = 0; k < kSteps; ++k) {
                            const uint64_t db = kDescHi64 | (b_lo + 2u * k);
                            const uint32_t accum = (kb | k) != 0 ? 1u : 0u;
                            const uint64_t da = kDescHi64 | (a_lo0 + kb * (kABlockBytes >> 4) + 2u * k);
                            if (kCG == 2) umma_f16_cg2(d_tmem, da, db, idesc, accum);
                            else          umma_f16(d_tmem, da, db, idesc, accum);
                        }
                        if (kCG == 2) umma_commit_cg2(&b_empty[bs]); else umma_commit(&b_empty[bs]);   // B stage reusable
                        if (++bs == static_cast<uint32_t>(p.b_stages)) { bs = 0; bph ^= 1; }
                    }
                    if (kCG == 2) umma_commit_cg2(&t_full[acc]); else umma_commit(&t_full[acc]);       // accumulator ready
                    acc ^= 1u; if (acc == 0u) tph ^= 1u;
                    ++t_it;
                }
                if (kCG == 2) umma_commit_cg2(&a_empty[as]); else umma_commit(&a_empty[as]);           // A stage reusable
                if (++as == static_cast<uint32_t>(p.a_stages)) { as = 0; aph ^= 1; }
            }
            if (pr) {
                p.prof[blockIdx.x * 32 + 4] = static_cast<unsigned long long>(clock64() - t_begin);
                p.prof[blockIdx.x * 32 + 5] = w_afull;
                p.prof[blockIdx.x * 32 + 6] = w_tempty;
                p.prof[blockIdx.x * 32 + 7] = w_bfull;
                p.prof[blockIdx.x * 32 + 8] = t_it;
            }
        }
        __syncwarp();
    } else if (kNorm && warp >= 2 + kEW) {
        // ===================== normaliser warps: fp32 rows -> L2-normalised fp16 rows in the workspace (K1 in-kernel) ====
        // Warp nw of 2 owns rows nw*4 .. nw*4+3 of every group of 8 rows of the CTA's tile; one row at a time per lane
        // set: lane l holds float4 #(l + 32 j) of the row (coalesced 512-byte loads, four rows = up to 8 KB in flight per
        // warp), warp-shuffle sum of squares, IEEE sqrt and one division per row, 8-byte fp16 stores.  The tiles are taken in
        // the order the TMA producer will load them; nothing else is waited for (the fp16 rows of different tiles are
        // different memory), so the warps run ahead of the tensor core by as much as their bandwidth allows.
        const int nw = warp - (2 + kEW);
        if (st32) {
            // ---- stage32 (dim_pad == 128): rows come out of the TMA-fed fp32 staging ring and go into the A stage as fp16 in the
            // K-major SWIZZLE_128B layout the MMA descriptors expect (row r of a K-block at r * 128 B, its 16-byte chunk c at
            // position c ^ (r & 7)) -- exactly what the TMA load of the fp16 workspace would have produced.  HBM sees each
            // candidate once, as fp32; there is no fp16 scratch and no K1 pass over the candidates whatever n_ref is.
            // ONE LANE PER ROW: a staging buffer is 32 rows as four 128-byte-wide swizzled column groups, so the eight lanes
            // of an LDS.128 / STS.128 wavefront hit eight different 16-byte bank groups on the way in and on the way out, and
            // there is no cross-lane reduction at all (the warp-per-row form spent its time in shuffles and in one
            // sqrt + division chain per row that the compiler will not interleave: 8-25 k cycles per tile; this is ~1.5 k).
            // The sum of squares runs in four interleaved chains (not warp_sum's tree): the fp16 rows can differ from the other
            // forms' by one fp16 ulp in rare elements, like x * (1/|x|) differs from K1's x / |x|.  The two warps take
            // alternate buffers.
            const bool pr = prof_on != nullptr && nw == 0;
            const long long t_nv_begin = clock64();
            uint32_t as = 0, aph = 0, n_done = 0;
            unsigned long long w_ae = 0, w_sf = 0, c_merge = 0;
            uint32_t g_buf = static_cast<uint32_t>(nw);                                   // staging buffers are numbered in load order
            const uint32_t sw = (static_cast<uint32_t>(lane) & 7u) << 4;                  // this row's swizzle term
            // ---- the epilogue's tail, run here: candidate tile u of this CTA (its state parked by the eight epilogue warps in
            // slot u & 1): each helper warp takes 64 rows, two per lane; merge the column halves (ties -> smaller index), emit.
            // rows of 68..96 floats: the fourth 32-float column group of every staging buffer is never loaded (a box that lies
            // entirely past `dim` is not issued); it is zeroed here once -- both warps write the same zeros, so each sees its own
            if (((p.dim + 31) >> 5) < 4) {
                for (int b = 0; b < p.s_bufs; ++b)
                    for (int i = lane; i < static_cast<int>(kStageBytes / 4 / 16); i += 32)
                        reinterpret_cast<uint4*>(smem_s + b * kStageBytes + 3 * (kStageBytes / 4))[i] = make_uint4(0u, 0u, 0u, 0u);
                __syncwarp();
            }
            bool k1_waited = false;
            auto merge_tile = [&](uint32_t u) {
                const long long tm0 = pr ? clock64() : 0;
                if (!k1_waited) {                                          // the list counters append_rows counts in are zeroed by K1
                    pdl_wait();
                    k1_waited = true;
                    if (blockIdx.x == 0 && nw == 0 && lane == 0) p.lists.hdr->refs_scanned = static_cast<int32_t>(n_ref);
                }
                const uint32_t slot = u & 1u;
                mbar_wait(&m_full[slot], (u >> 1) & 1u);
                const int64_t tile_u = tile0 + static_cast<int64_t>(u) * tile_stride;
                RowOut ro[2];
#pragma unroll
                for (int rr = 0; rr < 2; ++rr) {
                    const int r = nw * 64 + rr * 32 + lane;
                    const float* ma = merge + (slot * 2 + 0) * 11 * kTileM;
                    const float* mb = merge + (slot * 2 + 1) * 11 * kTileM;
                    Top3 t;
                    Hidden hid;
                    t.b1 = ma[0 * kTileM + r]; t.b2 = ma[1 * kTileM + r]; t.b3 = ma[2 * kTileM + r]; t.b4 = ma[3 * kTileM + r];
                    t.i1 = __float_as_int(ma[4 * kTileM + r]); t.i2 = __float_as_int(ma[5 * kTileM + r]); t.i3 = __float_as_int(ma[6 * kTileM + r]);
                    hid.amb = ma[7 * kTileM + r]; hid.amb2 = ma[8 * kTileM + r]; hid.base = __float_as_int(ma[9 * kTileM + r]);
                    hid.mask = __float_as_int(ma[10 * kTileM + r]);
                    const float o1 = mb[0 * kTileM + r], o2 = mb[1 * kTileM + r], o3 = mb[2 * kTileM + r], o4 = mb[3 * kTileM + r];
                    const int32_t j1 = __float_as_int(mb[4 * kTileM + r]), j2 = __float_as_int(mb[5 * kTileM + r]), j3 = __float_as_int(mb[6 * kTileM + r]);
                    Hidden hio;
                    hio.amb = mb[7 * kTileM + r]; hio.amb2 = mb[8 * kTileM + r];
                    hio.base = __float_as_int(mb[9 * kTileM + r]);
                    hio.mask = __float_as_int(mb[10 * kTileM + r]);
                    const HiddenM hm = hidden_merge(hid, hio);
                    if (o1 != -INFINITY) top3_merge_insert(t, o1, j1);
                    if (j2 >= 0) top3_merge_insert(t, o2, j2);
                    if (j3 >= 0) top3_merge_insert(t, o3, j3);
                    t.b4 = fmaxf(t.b4, o4);
                    ro[rr] = classify_row(p, t, hm, tile_u * (kTileM * kCG) + cta_rank * kTileM + r);
                }
                // the slot's contents are in registers: hand it back before the list appends (their atomics are the slow part)
                __syncwarp();
                if (lane == 0) mbar_arrive(&m_empty[slot]);
                append_rows<2>(p, ro, lane);
                if (pr) c_merge += static_cast<unsigned long long>(clock64() - tm0);
            };
            for (int64_t tile = tile0; tile < n_tiles; tile += tile_stride) {
                const int64_t row0 = tile * (kTileM * kCG) + cta_rank * kTileM;
                mbar_wait_timed(&a_empty[as], aph ^ 1, pr, w_ae);                          // A stage free again
                for (int part = nw; part < kTileM / kStageRows; part += 2, g_buf += 2) {
                    const uint32_t sb = g_buf % static_cast<uint32_t>(p.s_bufs);
                    const uint32_t sph = (g_buf / static_cast<uint32_t>(p.s_bufs)) & 1u;
                    mbar_wait_timed(&s_full[sb], sph, pr, w_sf);
                    const uint8_t* src = smem_s + sb * kStageBytes + lane * 128;
                    // ONE pass with the whole row (128 floats) in registers: 32 LDS.128 issued back to back, the sum of squares
                    // in four interleaved chains (not warp_sum's tree: the fp16 rows can differ from the other forms' by one fp16
                    // ulp in rare elements, like x * (1/|x|) differs from K1's x / |x|), one IEEE sqrt + division, then 16 STS.128.
                    // (Round 1 read every row twice in compact loops to keep the code small; with the tail's work moved into these
                    // warps their time per tile matters, and half the shared-memory reads is what pays.)
                    // Packed fp32 (FFMA2 / FMUL2, sm_100): the warp's time per buffer is its own instruction stream (ncu: one
                    // warp, IPC 0.34, two thirds of the instructions on the FMA pipe), so the 128 squares and the 128 scalings are
                    // issued two per instruction.  Products and the scaled values are the same IEEE results; the sum of squares is
                    // kept in eight partial sums instead of four (1 / |x| can differ in the last place from the earlier form).
                    float4 x[32];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const uint8_t* sg = src + g * (kStageBytes / 4);
#pragma unroll
                        for (int c = 0; c < 8; ++c)
                            x[g * 8 + c] = *reinterpret_cast<const float4*>(sg + ((static_cast<uint32_t>(c) << 4) ^ sw));
                    }
                    float2 q0 = make_float2(0.f, 0.f), q1 = q0, q2 = q0, q3 = q0;
#pragma unroll
                    for (int c = 0; c < 32; c += 2) {
                        const float2 a0 = make_float2(x[c].x, x[c].y), a1 = make_float2(x[c].z, x[c].w);
                        const float2 b0 = make_float2(x[c + 1].x, x[c + 1].y), b1 = make_float2(x[c + 1].z, x[c + 1].w);
                        q0 = __ffma2_rn(a0, a0, q0);
                        q1 = __ffma2_rn(a1, a1, q1);
                        q2 = __ffma2_rn(b0, b0, q2);
                        q3 = __ffma2_rn(b1, b1, q3);
                    }
                    const int r = part * kStageRows + lane;                               // row inside the tile
                    // rows past the end stay zero
                    const float qq = ((q0.x + q0.y) + (q1.x + q1.y)) + ((q2.x + q2.y) + (q3.x + q3.y));
                    const float inv = (row0 + r < p.n_cand) ? __fdiv_rn(1.0f, sqrtf(qq)) : 0.f;
                    const float2 inv2 = make_float2(inv, inv);
                    uint8_t* dst = smem_a + as * a_stage_bytes + r * 128;
#pragma unroll
                    for (int g = 0; g < 4; ++g) {                                         // 32 input floats -> 4 chunks of 8 halves
                        uint8_t* dg = dst + (g >> 1) * kABlockBytes;
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const float4 lo = x[g * 8 + 2 * c], hi = x[g * 8 + 2 * c + 1];
                            const float2 s0 = __fmul2_rn(make_float2(lo.x, lo.y), inv2), s1 = __fmul2_rn(make_float2(lo.z, lo.w), inv2);
                            const float2 s2 = __fmul2_rn(make_float2(hi.x, hi.y), inv2), s3 = __fmul2_rn(make_float2(hi.z, hi.w), inv2);
                            const __half2 h0 = __floats2half2_rn(s0.x, s0.y);
                            const __half2 h1 = __floats2half2_rn(s1.x, s1.y);
                            const __half2 h2 = __floats2half2_rn(s2.x, s2.y);
                            const __half2 h3 = __floats2half2_rn(s3.x, s3.y);
                            uint4 pk;
                            pk.x = *reinterpret_cast<const uint32_t*>(&h0);
                            pk.y = *reinterpret_cast<const uint32_t*>(&h1);
                            pk.z = *reinterpret_cast<const uint32_t*>(&h2);
                            pk.w = *reinterpret_cast<const uint32_t*>(&h3);
                            *reinterpret_cast<uint4*>(dg + ((static_cast<uint32_t>(4 * (g & 1) + c) << 4) ^ sw)) = pk;
                        }
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&s_empty[sb]);                             // the buffer can be refilled
                }
                fence_proxy_async_smem();                     // generic-proxy writes of the A tile -> visible to the MMAs (async proxy)
                __syncwarp();
                if (lane == 0) {
                    if (kCG == 2 && !leader) mbar_arrive_leader_cta(&a_full[as]);
                    else                     mbar_arrive(&a_full[as]);
                }
                // the A tile of candidate tile n_done is on its way to the tensor core; candidate tile n_done - 2 finished its
                // epilogue a whole tile ago: merge + emit it now, while the MMAs of tile n_done - 1 run
                if (kOffload && n_done >= 2u) merge_tile(n_done - 2u);
                ++n_done;
                if (++as == static_cast<uint32_t>(p.a_stages)) { as = 0; aph ^= 1; }
            }
            if (kOffload)
                // drain: the last two tiles (the very last one is merged by the epilogue warps themselves: inline_last)
                for (uint32_t u = n_done >= 2u ? n_done - 2u : 0u; u + 1u < n_done; ++u) merge_tile(u);
            if (pr && lane == 0) {
                p.prof[blockIdx.x * 32 + 13] = static_cast<unsigned long long>(clock64() - t_nv_begin);
                p.prof[blockIdx.x * 32 + 14] = n_done;
                p.prof[blockIdx.x * 32 + 18] = w_ae;
                p.prof[blockIdx.x * 32 + 19] = w_sf;
                p.prof[blockIdx.x * 32 + 20] = c_merge;
            }
        } else {
        const int nvec = p.dim >> 2;                                   // float4 per row (dim % 4 == 0 checked on the host)
        const int ld16 = p.kb_count * kBlockK;
        constexpr int kR = 4;                                         // rows in flight per warp
        constexpr uint32_t kNormAhead = 2;                            // tiles the warps may run ahead of the A loads
        const bool pr = prof_on != nullptr && nw == 0;
        const long long t_nv_begin = clock64();
        uint32_t n_done = 0;
        for (int64_t tile = tile0; tile < n_tiles; tile += tile_stride) {
            const int64_t row0 = tile * (kTileM * kCG) + cta_rank * kTileM;
            // at most two tiles ahead of the TMA loads: the fp16 rows then stay in L2 until they are consumed (running
            // free, the warps finished ALL tiles in a third of the kernel and every row made an HBM round trip)
            while (n_done >= ld_acquire_shared(cons_count) + kNormAhead) __nanosleep(200);
            // The fp16 rows are scratch: once a tile has been consumed nobody reads them again, and dropping the dirty L2
            // lines spares their write-back to HBM.  Passing the wait above means the A loads of tile n_done - 2 (or later)
            // have been issued, which needs that tile's A stage free, i.e. every MMA of tile n_done - 2 - a_stages retired --
            // and with them that tile's A loads.  (Done here, not by the TMA thread: 1024 discards per tile in the one
            // thread that feeds the B ring cost 7 % of the kernel.)
            if (n_done >= 2u + static_cast<uint32_t>(p.a_stages)) {
                const int64_t old_tile = tile - static_cast<int64_t>(2 + p.a_stages) * tile_stride;
                const int64_t old_row0 = old_tile * (kTileM * kCG) + cta_rank * kTileM;
                const int64_t bytes = static_cast<int64_t>(kTileM) * ld16 * 2;          // a full tile: it is not the last one
                const char* base = reinterpret_cast<const char*>(p.cand16) + old_row0 * ld16 * 2;
                for (int64_t off = static_cast<int64_t>(nw * 32 + lane) * 128; off + 128 <= bytes; off += 64 * 128)
                    asm volatile("discard.global.L2 [%0], 128;" ::"l"(base + off) : "memory");
            }
            for (int rb = nw * kR; rb < kTileM; rb += 2 * kR) {
                if (row0 + rb >= p.n_cand) break;
                float4 v[kR][4];
#pragma unroll
                for (int u = 0; u < kR; ++u) {
                    int64_t gr = row0 + rb + u;
                    gr = gr < p.n_cand ? gr : p.n_cand - 1;            // clamped: loads stay unconditional and in flight together
                    const float4* src = reinterpret_cast<const float4*>(p.cand32 + gr * p.dim);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int f = lane + 32 * j;
                        v[u][j] = f < nvec ? ldg_stream_evict_first_f4(src + f) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
#pragma unroll
                for (int u = 0; u < kR; ++u) {
                    const int64_t gr = row0 + rb + u;
                    float ss = 0.f;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        ss = fmaf(v[u][j].x, v[u][j].x, ss); ss = fmaf(v[u][j].y, v[u][j].y, ss);
                        ss = fmaf(v[u][j].z, v[u][j].z, ss); ss = fmaf(v[u][j].w, v[u][j].w, ss);
                    }
                    ss = warp_sum(ss);
                    // one IEEE division per row, then multiplies: 16 division sequences per row and lane made these two warps
                    // ALU bound (118 k cycles per 128 x 512 tile).  <= 1.5 ulp from K1's x / |x| before the fp16 rounding.
                    const float inv = __fdiv_rn(1.0f, sqrtf(ss));
                    if (gr < p.n_cand) {
                        __half* dst = p.cand16 + gr * ld16;
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int f = lane + 32 * j;
                            if (4 * f < ld16) {                        // columns [dim, ld16) are the zero K padding
                                uint2 pk = make_uint2(0u, 0u);
                                if (f < nvec) {
                                    const __half2 h0 = __floats2half2_rn(v[u][j].x * inv, v[u][j].y * inv);
                                    const __half2 h1 = __floats2half2_rn(v[u][j].z * inv, v[u][j].w * inv);
                                    pk.x = *reinterpret_cast<const uint32_t*>(&h0);
                                    pk.y = *reinterpret_cast<const uint32_t*>(&h1);
                                }
                                reinterpret_cast<uint2*>(dst)[f] = pk;
                            }
                        }
                    }
                }
            }
            fence_proxy_async_global();                                 // generic-proxy stores -> visible to the TMA loads
            __syncwarp();
            if (lane == 0) red_release_shared_add(&norm_count[nw], 1u);
            ++n_done;
        }
        if (pr && lane == 0) {
            p.prof[blockIdx.x * 32 + 13] = static_cast<unsigned long long>(clock64() - t_nv_begin);
            p.prof[blockIdx.x * 32 + 14] = n_done;
        }
        }   // !st32
    } else {
        // ===================== epilogue: one thread per (candidate row, column half) =====================
        const int q = warp & 3;                               // TMEM lane quadrant this warp may access
        const int h = (warp - 2) >> 2;                        // column part of every reference tile this warp scans
        const int r_in_tile = q * 32 + lane;
        uint32_t t_it = 0, c_it = 0;                          // reference tiles / candidate tiles this CTA has finished
        constexpr bool kAlt = kParts == 2;                    // the two column parts take turns at the merge + emit tail
        bool first_tile = true;
        const bool pr = prof_on != nullptr && warp == 4;                 // one part-0 warp reports
        unsigned long long w_tfull = 0, c_hot = 0, c_gen = 0, c_bar1 = 0, c_tail = 0;
        // the score dump only exists in the general loop
        const bool hot_ok = !kInstr || p.dbg_scores == nullptr;
        // the two epilogue policies: compile-time constants in the production instantiations
        const bool grid_updates = kAlways == 2 ? p.grid_updates != 0 : kAlways == 1;     // unconditional update path
        const bool grid_exact = kExact == 2 ? p.grid_exact != 0 : kExact == 1;           // several in-window columns in one part: exact masks, or flag the row
        const long long t_begin = clock64();
        for (int64_t tile = tile0; tile < n_tiles; tile += tile_stride) {
            Top3 t;
            t.b1 = t.b2 = t.b3 = t.b4 = -INFINITY;
            t.i1 = 0;
            t.i2 = t.i3 = -1;
            float gate = -INFINITY;                             // running best - delta
            Hidden hid;                                         // see struct Hidden
            hid.amb = hid.amb2 = -INFINITY;
            hid.base = 0;
            hid.mask = 0;
            const int64_t row = tile * (kTileM * kCG) + cta_rank * kTileM + r_in_tile;
            // kSelf: this row's global index g; the masked body sets columns >= self_lim (past the last reference, or from g on
            // in FFR_SELF_EARLIER) and column g to -inf
            const int32_t self_g = kSelf ? static_cast<int32_t>(p.self_row0 + row) : 0;
            const int32_t self_lim = kSelf ? (p.self_mode == FFR_SELF_EARLIER ? self_g : static_cast<int32_t>(n_ref)) : 0;
            float delta_row = 0.f, s_row = 0.f;
            if constexpr (kEuclid) {
                static_assert(kNormMode == 0 && !kInstr, "Euclid runs on the K1 schedule, production build only");
                // K1 writes the scales; it precedes this kernel as its programmatic dependency
                if (first_tile) pdl_wait();
                s_row = row < p.n_cand ? __ldg(p.cand_scale + row) : 0.f;
                // |score error| <= fp16 operand error (delta, as for cosine) + a few fp32 roundings of the bias term (beta and
                // 1/|c| each carry one, the FFMA another): 8 ulp of max |beta| / |c| covers them.  (A zero-norm or non-finite row
                // -- s_row not finite -- gets a NaN window here and goes to the full fp32 rescan in the tail.)
                delta_row = fmaf(__ldg(p.bias_max) * s_row, 4.76837158e-7f, p.delta);
            }
            // One reference tile.  The loop over FULL tiles and the one partial last tile are separate copies of this body: the
            // masking of columns >= n_ref is 260 instructions that the hot loop would otherwise carry (and jump over) on every
            // tile -- the body is what has to stream through the instruction cache.
            auto ref_tile = [&](const int rt, auto partial_tag) {
                constexpr bool kPartial = decltype(partial_tag)::value;
                const uint32_t acc = t_it & 1, tph = (t_it >> 1) & 1;
                mbar_wait_timed(&t_full[acc], tph, pr, w_tfull);
                const long long tp0 = pr ? clock64() : 0;
                tc_fence_after();
                const int32_t col0 = rt * kAccN;
                const int64_t ncols64 = n_ref - static_cast<int64_t>(col0);
                const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * kAccN + h * (kChunksPerPart * 32);
                const int32_t base0 = col0 + h * (kChunksPerPart * 32);
                if (hot_ok) {
                    // ---- hot loop: straight-line code.  All of this warp's columns are
                    // pulled out of TMEM back to back, the accumulator stage goes back to the MMA warp at once, then
                    // one max tree per 32-column chunk and ONE branch per tile guards the update path.  A taken branch
                    // costs ~30 cycles here (two warps per scheduler cannot hide the refetch): the loop shape, not the
                    // arithmetic, was what bounded the epilogue before (tools/epi_bench.cu).
                    float v[kChunksPerPart][32];
#pragma unroll
                    for (int cc = 0; cc < kChunksPerPart; ++cc) tmem_ld_32x32(taddr + cc * 32, v[cc]);
                    tmem_ld_wait();
#pragma unroll
                    for (int cc = 0; cc < kChunksPerPart; ++cc) tmem_ld_fence(v[cc]);
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if (kCG == 2 && !leader) mbar_arrive_leader_relaxed(&t_empty[acc]);
                        else                     mbar_arrive(&t_empty[acc]);
                    }
                    if constexpr (kEuclid) {                       // score = acc + beta_col / |c|, two columns per FFMA2
                        const float4* bp = reinterpret_cast<const float4*>(p.ref_bias + base0);
                        const float2 s2 = make_float2(s_row, s_row);
#pragma unroll
                        for (int cc = 0; cc < kChunksPerPart; ++cc)
#pragma unroll
                            for (int j4 = 0; j4 < 8; ++j4) {
                                const float4 b = __ldg(bp + cc * 8 + j4);
                                const float2 lo = __ffma2_rn(make_float2(b.x, b.y), s2, make_float2(v[cc][4 * j4], v[cc][4 * j4 + 1]));
                                const float2 hi = __ffma2_rn(make_float2(b.z, b.w), s2, make_float2(v[cc][4 * j4 + 2], v[cc][4 * j4 + 3]));
                                v[cc][4 * j4] = lo.x; v[cc][4 * j4 + 1] = lo.y; v[cc][4 * j4 + 2] = hi.x; v[cc][4 * j4 + 3] = hi.y;
                            }
                    }
                    if constexpr (kSelf) {
                        if constexpr (kPartial) {                  // masked body of self mode (after the Euclid bias)
#pragma unroll
                            for (int cc = 0; cc < kChunksPerPart; ++cc)
#pragma unroll
                                for (int j = 0; j < 32; ++j) {
                                    const int32_t c = base0 + cc * 32 + j;
                                    v[cc][j] = (c >= self_lim || c == self_g) ? -INFINITY : v[cc][j];
                                }
                        }
                    } else if constexpr (kPartial) {               // partial last reference tile: columns >= n_ref -> -inf
                        const int n_left = static_cast<int>(ncols64) - h * (kChunksPerPart * 32);
#pragma unroll
                        for (int cc = 0; cc < kChunksPerPart; ++cc)
                            if (n_left - cc * 32 < 32) mask_chunk(v[cc], n_left - cc * 32);
                    }
                    float cm[kChunksPerPart], sx[kChunksPerPart][4];
#pragma unroll
                    for (int cc = 0; cc < kChunksPerPart; ++cc) {
                        group_max8(v[cc], sx[cc]);
                        cm[cc] = fmax3(sx[cc][0], sx[cc][1], fmaxf(sx[cc][2], sx[cc][3]));
                    }
                    float m = cm[0];
#pragma unroll
                    for (int cc = 1; cc < kChunksPerPart; ++cc) m = fmaxf(m, cm[cc]);
                    // short reference sets: some lane of the warp sets a record on nearly every tile, so the update runs
                    // unconditionally and branch-free; long ones: behind one branch on the part maximum.  (Round-1c's
                    // per-chunk update paths are gone from this loop: dead code in it costs wall clock.)
                    if (grid_updates || m >= gate) update_grid<kChunksPerPart>(v, sx, cm, m, base0, kEuclid ? delta_row : p.delta, grid_exact, t, gate, hid);
                    if (pr) c_hot += static_cast<unsigned long long>(clock64() - tp0);
                } else {
                    // ---- general loop, one chunk at a time: the score dump only
                    const int ncols = ncols64 > kAccN ? kAccN : static_cast<int>(ncols64);
                    const int n_left = ncols - h * (kChunksPerPart * 32);             // live columns of this warp's part
                    float va[32];
                    for (int cc = 0; cc < kChunksPerPart && cc * 32 < n_left; ++cc) {
                        tmem_ld_32x32(taddr + cc * 32, va);
                        tmem_ld_wait();
                        tmem_ld_fence(va);
                        if (n_left - cc * 32 < 32) mask_chunk(va, n_left - cc * 32);
                        if (p.dbg_scores != nullptr && row < p.n_cand) {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (base0 + cc * 32 + j < p.n_ref) p.dbg_scores[row * p.n_ref + base0 + cc * 32 + j] = va[j];
                        }
                        const float cmx = chunk_max(va);
                        if (cmx >= gate) update_chunk(va, cmx, base0 + cc * 32, p.delta, t, gate, hid.amb2);
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if (kCG == 2 && !leader) mbar_arrive_leader_relaxed(&t_empty[acc]);
                        else                     mbar_arrive(&t_empty[acc]);
                    }
                    if (pr) c_gen += static_cast<unsigned long long>(clock64() - tp0);
                }
                ++t_it;
            };
            const int32_t n_full = static_cast<int32_t>(n_ref / kAccN);
            if constexpr (kSelf) {
                // the masked body runs on the partial last tile and on every tile that holds a row of this CTA pair's candidate
                // tile (two tiles when the rows straddle a tile boundary: row_begin not a multiple of 256); once per (candidate
                // tile, reference tile), from the indices alone
                const int64_t g0 = p.self_row0 + tile * (kTileM * kCG);
                const int64_t g1 = p.self_row0 + (tile * (kTileM * kCG) + (kTileM * kCG - 1) < p.n_cand
                                                      ? tile * (kTileM * kCG) + (kTileM * kCG - 1) : p.n_cand - 1);
                const int32_t rt_end = self_rt_end(p, tile, n_rt);
                for (int rt = 0; rt < rt_end; ++rt) {
                    const int64_t c0 = static_cast<int64_t>(rt) * kAccN;
                    if (rt >= n_full || (c0 <= g1 && c0 + kAccN > g0)) ref_tile(rt, std::true_type{});
                    else                                               ref_tile(rt, std::false_type{});
                }
            }
            for (int rt = 0; rt < (kSelf ? 0 : n_full); ++rt) ref_tile(rt, std::false_type{});
            if (!kSelf && n_full < n_rt) ref_tile(n_full, std::true_type{});
            // ---- hand the other column part(s) over, merge, emit.  The merging thread runs ~300 dependent instructions
            // alone on its scheduler (its partner is already in the next tile's loads), so with two parts the ROLE alternates
            // from candidate tile to candidate tile: each warp carries the tail every other tile, and since the reader of
            // tile n is the writer of tile n + 1 the buffer needs no "free again" barrier.  Named barriers couple only the
            // warps of ONE lane quadrant (ids 1+q / 5+q, alternating with the tile parity so that an early arrive for tile
            // n + 2 cannot complete tile n's barrier); with CTA-wide barriers every quadrant waited for the slowest warp.
            const long long t_tail0 = pr ? clock64() : 0;
            // ... except for the CTA's LAST candidate tile: nothing is left to overlap its tail with, and four merger warps (32 rows
            // each) finish it in half the time the two helper warps (64 rows each) need -- the kernel's drain.
            const bool inline_last = kOffload && tile + tile_stride >= n_tiles;
            if (kOffload && !inline_last) {
                // stage32 with several reference tiles per candidate tile: the tail is NOT run here.  Merging the two column halves, classifying the row and appending to K3's
                // lists is ~300 dependent instructions that used to stall this warp for as long as a reference tile's hot loop
                // (with four reference tiles per candidate tile -- BASELINE configs[1] -- a fifth of the epilogue's time).  Both
                // halves park their state in one of two shared-memory slots and go on with the next candidate tile; the two
                // normaliser warps (helpers), which have spare time at every reference-set size, merge and emit it.
                const uint32_t slot = c_it & 1u;
                mbar_wait(&m_empty[slot], ((c_it >> 1) & 1u) ^ 1u);          // merged two candidate tiles ago: free again
                float* mg = merge + (slot * 2 + h) * 11 * kTileM;
                mg[0 * kTileM + r_in_tile] = t.b1;
                mg[1 * kTileM + r_in_tile] = t.b2;
                mg[2 * kTileM + r_in_tile] = t.b3;
                mg[3 * kTileM + r_in_tile] = t.b4;
                mg[4 * kTileM + r_in_tile] = __int_as_float(t.i1);
                mg[5 * kTileM + r_in_tile] = __int_as_float(t.i2);
                mg[6 * kTileM + r_in_tile] = __int_as_float(t.i3);
                mg[7 * kTileM + r_in_tile] = hid.amb;
                mg[8 * kTileM + r_in_tile] = hid.amb2;
                mg[9 * kTileM + r_in_tile] = __int_as_float(hid.base);
                mg[10 * kTileM + r_in_tile] = __int_as_float(hid.mask);
                __syncwarp();
                if (lane == 0) mbar_arrive(&m_full[slot]);                  // (release at CTA scope: the warp's stores above)
            } else {
            float* xmerge = merge;                               // exchange buffer of the two column halves
            if (kOffload) {
                // (the parked-state slot this tile would have used, once the helper warps have emptied it)
                const uint32_t slot = c_it & 1u;
                mbar_wait(&m_empty[slot], ((c_it >> 1) & 1u) ^ 1u);
                xmerge = merge + slot * 2 * 11 * kTileM;
                pdl_wait();
                if (blockIdx.x == 0 && threadIdx.x == 64) p.lists.hdr->refs_scanned = static_cast<int32_t>(n_ref);   // (a CTA with ONE tile: the helper warps never merge)
            } else if (first_tile) {
                pdl_wait();                                      // the re-check header the appends below count in is zeroed by K1
                if (blockIdx.x == 0 && threadIdx.x == 64) p.lists.hdr->refs_scanned = static_cast<int32_t>(n_ref);
            }
            const bool merger = kAlt ? (((c_it ^ static_cast<uint32_t>(h)) & 1u) == 0u) : (h == 0);
            const uint32_t bar_ready = kAlt ? (1 + q + 4 * (c_it & 1u)) : (1 + q);
            if (!merger) {
                float* mg = xmerge + (kAlt ? 0 : (h - 1) * 11 * kTileM);
                if (!kAlt && !first_tile) named_bar_sync(5 + q, kParts * 32);  // merge buffer free again
                mg[0 * kTileM + r_in_tile] = t.b1;
                mg[1 * kTileM + r_in_tile] = t.b2;
                mg[2 * kTileM + r_in_tile] = t.b3;
                mg[3 * kTileM + r_in_tile] = t.b4;
                mg[4 * kTileM + r_in_tile] = __int_as_float(t.i1);
                mg[5 * kTileM + r_in_tile] = __int_as_float(t.i2);
                mg[6 * kTileM + r_in_tile] = __int_as_float(t.i3);
                mg[7 * kTileM + r_in_tile] = hid.amb;
                mg[8 * kTileM + r_in_tile] = hid.amb2;
                mg[9 * kTileM + r_in_tile] = __int_as_float(hid.base);
                mg[10 * kTileM + r_in_tile] = __int_as_float(hid.mask);
                __threadfence_block();
                named_bar_arrive(bar_ready, kParts * 32);
            } else {
                const long long tm0 = pr ? clock64() : 0;
                named_bar_sync(bar_ready, kParts * 32);
                if (pr) c_bar1 += static_cast<unsigned long long>(clock64() - tm0);
                float ob[kParts - 1][4];
                int32_t oi[kParts - 1][3];
                static_assert(kParts == 2, "hidden_merge joins the states of TWO column halves");
                HiddenM hm = hidden_single(hid);
#pragma unroll
                for (int pp = 0; pp < kParts - 1; ++pp) {
                    const float* mg = xmerge + pp * 11 * kTileM;
#pragma unroll
                    for (int e = 0; e < 4; ++e) ob[pp][e] = mg[e * kTileM + r_in_tile];
#pragma unroll
                    for (int e = 0; e < 3; ++e) oi[pp][e] = __float_as_int(mg[(4 + e) * kTileM + r_in_tile]);
                    // the other half's hidden-column state (hidden_merge: adjacent parts are joined, else the larger maximum leads)
                    Hidden hio;
                    hio.amb = mg[7 * kTileM + r_in_tile]; hio.amb2 = mg[8 * kTileM + r_in_tile];
                    hio.base = __float_as_int(mg[9 * kTileM + r_in_tile]);
                    hio.mask = __float_as_int(mg[10 * kTileM + r_in_tile]);
                    hm = hidden_merge(hid, hio);
                }
                if (!kAlt) named_bar_arrive(5 + q, kParts * 32);
#pragma unroll
                for (int pp = 0; pp < kParts - 1; ++pp) {
                    if (ob[pp][0] != -INFINITY) top3_merge_insert(t, ob[pp][0], oi[pp][0]);
                    if (oi[pp][1] >= 0) top3_merge_insert(t, ob[pp][1], oi[pp][1]);
                    if (oi[pp][2] >= 0) top3_merge_insert(t, ob[pp][2], oi[pp][2]);
                    t.b4 = fmaxf(t.b4, ob[pp][3]);
                }

                RowOut ro[1];
                ro[0] = classify_row<kEuclid, kSelf>(p, t, hm, row, delta_row, !(fabsf(s_row) <= 3.4e38f),
                                                     kSelf && p.self_mode == FFR_SELF_EARLIER && self_g == 0);
                append_rows<1>(p, ro, lane);
            }
            }   // !st32
            first_tile = false;
            ++c_it;
            if (pr) c_tail += static_cast<unsigned long long>(clock64() - t_tail0);
        }
        if (pr && lane == 0) {
            p.prof[blockIdx.x * 32 + 16] = c_bar1;
            p.prof[blockIdx.x * 32 + 17] = c_tail;
            p.prof[blockIdx.x * 32 + 10] = static_cast<unsigned long long>(clock64() - t_begin);
            p.prof[blockIdx.x * 32 + 11] = w_tfull;
            p.prof[blockIdx.x * 32 + 3] = c_hot;
            (void)c_gen;
        }
        // balance the last bar.arrive(5 + q) of the lower part so no barrier state is left pending
        if (!kAlt && h != 0 && !first_tile) named_bar_sync(5 + q, kParts * 32);
    }

    tc_fence_before();
    if (kCG == 2) cluster_sync_all(); else __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        if (kCG == 2) tmem_dealloc_cg2<kTmemCols>(tmem_base);
        else          tmem_dealloc<kTmemCols>(tmem_base);
    }
    if (prof_on != nullptr && threadIdx.x == 0) {
        unsigned long long ts;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ts));
        p.prof[blockIdx.x * 32 + 9] = ts;                              // ns: CTA exit
    }
}

// ---- host side -----------------------------------------------------------------------------------

// cuTensorMapEncodeTiled is pure host arithmetic (~1 us): a launch-bound caller (BASELINE configs[1]: ~25 us of GPU work per
// call) repeats the same (pointer, shape) every step, so the last few encodings are kept per thread.
struct TmapSlot { const void* base; int64_t rows; int32_t ld, box_cols, box_rows, kind; CUtensorMap map; bool valid; };
thread_local TmapSlot g_tmaps[6];
thread_local int g_tmap_next = 0;
const CUtensorMap* tmap_lookup(const void* base, int64_t rows, int32_t ld, int32_t box_cols, int32_t box_rows, int kind) {
    for (const TmapSlot& t : g_tmaps)
        if (t.valid && t.base == base && t.rows == rows && t.ld == ld && t.box_cols == box_cols && t.box_rows == box_rows && t.kind == kind)
            return &t.map;
    return nullptr;
}
void tmap_store(const void* base, int64_t rows, int32_t ld, int32_t box_cols, int32_t box_rows, int kind, const CUtensorMap& m) {
    TmapSlot& t = g_tmaps[g_tmap_next];
    g_tmap_next = (g_tmap_next + 1) % 6;
    t.base = base; t.rows = rows; t.ld = ld; t.box_cols = box_cols; t.box_rows = box_rows; t.kind = kind; t.map = m; t.valid = true;
}


typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static std::atomic<EncodeTiledFn> fn{nullptr};
    EncodeTiledFn f = fn.load(std::memory_order_acquire);
    if (f == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            return nullptr;
        f = reinterpret_cast<EncodeTiledFn>(p);
        fn.store(f, std::memory_order_release);
    }
    return f;
}

// fp16 matrix [rows, ld] row-major, box = [box_rows, 64 cols], 128-byte swizzle, zero fill out of bounds
int make_tmap(CUtensorMap* m, const __half* base, int64_t rows, int32_t ld, int32_t box_rows) {
    if (const CUtensorMap* c = tmap_lookup(base, rows, ld, kBlockK, box_rows, 16)) { *m = *c; return FFR_OK; }
    EncodeTiledFn fn = get_encode_fn();
    if (fn == nullptr) { set_error("cuTensorMapEncodeTiled entry point not available (driver too old / no GPU)"); return FFR_ERR_CUDA; }
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(ld), static_cast<cuuint64_t>(rows)};
    cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * 2};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(kBlockK), static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), gdim, gstride, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed: CUresult %d (rows=%lld ld=%d)", (int)r, (long long)rows, ld); return FFR_ERR_CUDA; }
    tmap_store(base, rows, ld, kBlockK, box_rows, 16, *m);
    return FFR_OK;
}

// fp32 matrix [rows, dim] row-major (pitch dim * 4 bytes), box = [box_rows, 32 floats = 128 bytes], 128-byte swizzle, zero
// fill out of bounds (column groups >= dim, rows past the end)
int make_tmap_f32(CUtensorMap* m, const float* base, int64_t rows, int32_t dim, int32_t box_cols, int32_t box_rows) {
    if (const CUtensorMap* c = tmap_lookup(base, rows, dim, box_cols, box_rows, 32)) { *m = *c; return FFR_OK; }
    EncodeTiledFn fn = get_encode_fn();
    if (fn == nullptr) { set_error("cuTensorMapEncodeTiled entry point not available (driver too old / no GPU)"); return FFR_ERR_CUDA; }
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(dim), static_cast<cuuint64_t>(rows)};
    cuuint64_t gstride[1] = {static_cast<cuuint64_t>(dim) * 4};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (fp32) failed: CUresult %d (rows=%lld dim=%d)", (int)r, (long long)rows, dim); return FFR_ERR_CUDA; }
    tmap_store(base, rows, dim, box_cols, box_rows, 32, *m);
    return FFR_OK;
}

// stage32 handles rows of 68..128 floats (dim_pad == 128; dim % 4 == 0 is already a condition of fusing)
bool filter_mma_stage32_ok(int32_t dim, int32_t dim_pad) {
    return dim_pad == 128 && (dim % 4) == 0 && knobs().stage32 != 0;
}

std::atomic<unsigned long long*> g_prof{nullptr};          // diagnostics buffer (ffr_debug_set_prof)

// what the last launch of this thread looked like (test hook ffr_debug_last_k2_config)
thread_local int g_last_cfg[8] = {0, 0, 0, 0, 0, 0, 0, 0};

int a_stage_count(int32_t dim_pad) {
    const uint32_t a_stage = (dim_pad / kBlockK) * kABlockBytes;
    return a_stage <= 32768 ? 3 : (a_stage <= 65536 ? 2 : 1);
}

struct BandArgs { float tol; int32_t* count; int64_t* rows; int64_t cap; };

// cand32 != nullptr: the candidates' normalisation runs inside the kernel, which then WRITES cand16 (workspace) itself
int launch_filter_mma_impl(const __half* ref16, int64_t n_ref, __half* cand16, const float* cand32, int32_t dim,
                           int64_t n_cand, int32_t dim_pad,
                           float thr, float delta, float thr_band, int64_t ref_index_base, uint8_t* keep, int32_t* idx, float* val,
                           RecheckLists lists, int no_recheck, BandArgs band, float* dbg_scores, bool after_k1,
                           const int32_t* ref_map, const int32_t* n_ref_dev, cudaStream_t s,
                           const float* euclid_bias, const float* cand_scale, const float* bias_max, SelfArgs self) {
    if (dim_pad % kBlockK != 0 || dim_pad < kBlockK || dim_pad > 512) {
        set_error("filter_mma: padded dim %d not in {64..512 step 64}", dim_pad);
        return FFR_ERR_UNSUPPORTED;
    }
    if (n_ref >= (int64_t(1) << 31) - 512 || n_cand >= (int64_t(1) << 31) - 512) {
        set_error("filter_mma: n_ref / n_cand must be < 2^31");
        return FFR_ERR_UNSUPPORTED;
    }
    const Knobs& kn = knobs();                         // FFR_* dispatch overrides, read once per process (DESIGN.md §10)
    const int sms = num_sms();
    // cta_group::2 everywhere: half the B bytes per SM and 8 KB instead of 12 KB of shared-memory operand reads per MMA
    // (measured: dim 128 1292 vs 1152 TFLOP/s, dim 256 1207 vs 1010, dim 512 1429 vs 1212)
    int cg = kn.cta_group;
    if (cg != 2 || (sms & 1)) cg = 1;
    const bool fuse = cand32 != nullptr;
    const bool euclid = euclid_bias != nullptr;
    if (euclid && (cg != 2 || fuse || no_recheck || dbg_scores != nullptr)) {
        set_error("filter_mma: the Euclid kernel exists for cta_group::2, the K1 schedule and the re-checked build only");
        return FFR_ERR_UNSUPPORTED;
    }
    const bool self_mode = self.mode >= 0;
    if (self_mode && (cg != 2 || fuse || no_recheck || dbg_scores != nullptr || n_ref_dev != nullptr)) {
        set_error("filter_mma: the self-mode kernel exists for cta_group::2, the K1 schedule and the re-checked build only");
        return FFR_ERR_UNSUPPORTED;
    }
    const int kb = dim_pad / kBlockK;
    constexpr int acc_n = kTileN;
    const uint32_t a_stage = kb * kABlockBytes;
    const uint32_t b_stage = (acc_n / cg) * kBlockK * 2;
    int a_stages = a_stage_count(dim_pad);
    constexpr int ew = 8;                                  // epilogue warps: 4 TMEM lane quadrants x 2 column halves
    // stage32 (fused normalisation, 128-d rows): fp32 rows staged by TMA, two A stages (the normaliser fills one while the
    // MMAs read the other), the B ring gets what is left (>= 2 stages); the tail's hand-over buffer is two slots x two halves
    const bool st32 = fuse && filter_mma_stage32_ok(dim, dim_pad);
    // (FFR_TAIL_OFFLOAD: -1 auto = offload from two reference tiles per candidate tile up, 0 / 1 force)
    const bool offload = st32 && (kn.tail_offload >= 0 ? kn.tail_offload != 0 : n_ref > kTileN);
    const uint32_t extra = kBarrierBytes + (offload ? 4 : 1) * kMergeBytes;
    int s_bufs = st32 ? (offload ? kMaxSBufs - 1 : kMaxSBufs) : 0;   // (with the merge slots: five 16 KB staging buffers leave three B stages)
    if (st32) {
        a_stages = 2;
        while (s_bufs > 3 && kSmemLimit - extra - s_bufs * kStageBytes < a_stages * a_stage + 2 * b_stage) --s_bufs;
    }
    const uint32_t budget = kSmemLimit - extra - s_bufs * kStageBytes;
    while (a_stages > 1 && a_stages * a_stage + 2 * b_stage > budget) --a_stages;
    if (a_stages * a_stage + 2 * b_stage > budget) { set_error("filter_mma: not enough shared memory for dim %d", dim_pad); return FFR_ERR_UNSUPPORTED; }
    int b_stages = static_cast<int>((budget - a_stages * a_stage) / b_stage);
    if (b_stages > kMaxBStages) b_stages = kMaxBStages;
    const uint32_t smem = a_stages * a_stage + b_stages * b_stage + s_bufs * kStageBytes + extra;

    CUtensorMap tm_c, tm_r;
    int rc = make_tmap(&tm_r, ref16, n_ref, dim_pad, acc_n / cg);
    if (rc != FFR_OK) return rc;
    if (st32) {
        tm_c = tm_r;                                           // (unused placeholder: stage32 has no fp16 candidate matrix)
    } else {
        rc = make_tmap(&tm_c, cand16, n_cand, dim_pad, kTileM);
        if (rc != FFR_OK) return rc;
    }
    CUtensorMap tm_c32 = tm_r;                                 // (unused placeholder unless stage32)
    if (st32) {
        rc = make_tmap_f32(&tm_c32, cand32, n_cand, dim, 32, kStageRows);
        if (rc != FFR_OK) return rc;
    }

    unsigned long long* const prof = g_prof.load(std::memory_order_relaxed);
    KParams p;
    p.n_ref = n_ref; p.n_ref_dev = n_ref_dev; p.ref_map = ref_map; p.n_cand = n_cand; p.kb_count = kb; p.a_stages = a_stages; p.b_stages = b_stages;
    p.thr = thr; p.delta = delta; p.thr_band = thr_band; p.ref_index_base = ref_index_base;
    p.keep = keep; p.best_idx = idx; p.best_val = val; p.lists = lists; p.no_recheck = no_recheck; p.dbg_scores = dbg_scores; p.prof = prof;
    p.band_tol = band.tol; p.band_count = no_recheck ? band.count : nullptr; p.band_rows = band.rows; p.band_cap = band.cap;
    p.ref_bias = euclid_bias; p.cand_scale = cand_scale; p.bias_max = bias_max;
    p.self_row0 = self.row0; p.self_mode = self.mode;
    p.cand32 = cand32; p.cand16 = cand16; p.dim = dim;
    p.stage32 = st32 ? 1 : 0;
    p.s_bufs = s_bufs;
    p.grid_updates = n_ref <= kn.grid_update_refs ? 1 : 0;
    // The flag-only form hands every same-part near tie to K3, which rescans the 128 references of that part in fp32 (round
    // 1 rescanned ALL references, which only paid for 128-d x >= 32 k references).  It RELIES on K3: without the re-check
    // (fp16 input, FFR_FLAG_NO_RECHECK, the score dump) the placeholder index it inserts would be the final answer, so those
    // callers always get the exact per-column masks (FFR_GRID_EXACT=1 forces them everywhere).
    p.grid_exact = kn.grid_exact >= 0 ? kn.grid_exact : 0;
    if (no_recheck || dbg_scores != nullptr) p.grid_exact = 1;
    if (euclid || self_mode) p.grid_exact = 0;             // (K3 always runs behind the Euclid and the self-mode kernels)

    typedef void (*KernelFn)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const KParams);
    // Instantiations: cta_group::2 production kernels carry the two epilogue policies as compile-time constants (no dead
    // fall-back code in the hot loop); the instrumented build (tools/diag_mma.py, the tests' score dump) and the
    // cta_group::1 fall-back (odd SM counts, FFR_CTA_GROUP=1) read them at run time.
    const bool instr = prof != nullptr || dbg_scores != nullptr;
    const int nm = st32 ? (offload ? 2 : 3) : (fuse ? 1 : 0);
#define FFR_K(CG, NM, E, A, I) filter_mma_kernel<CG, NM, E, A, I>
#define FFR_K_POLICY(NM) {FFR_K(2, NM, 0, 0, false), FFR_K(2, NM, 0, 1, false), FFR_K(2, NM, 1, 0, false), FFR_K(2, NM, 1, 1, false)}
    static const KernelFn prod2[4][4] = {FFR_K_POLICY(0), FFR_K_POLICY(1), FFR_K_POLICY(2), FFR_K_POLICY(3)};
    static const KernelFn instr2[4] = {FFR_K(2, 0, 2, 2, true), FFR_K(2, 1, 2, 2, true), FFR_K(2, 2, 2, 2, true), FFR_K(2, 3, 2, 2, true)};
    static const KernelFn prod1[4] = {FFR_K(1, 0, 2, 2, false), FFR_K(1, 1, 2, 2, false), FFR_K(1, 2, 2, 2, false), FFR_K(1, 3, 2, 2, false)};
    static const KernelFn instr1[4] = {FFR_K(1, 0, 2, 2, true), FFR_K(1, 1, 2, 2, true), FFR_K(1, 2, 2, 2, true), FFR_K(1, 3, 2, 2, true)};
#undef FFR_K_POLICY
#undef FFR_K
    static const KernelFn euclid2[2] = {filter_mma_kernel<2, 0, 0, 0, false, true>, filter_mma_kernel<2, 0, 0, 1, false, true>};
    static const KernelFn self2[2][2] = {{filter_mma_kernel<2, 0, 0, 0, false, false, true>, filter_mma_kernel<2, 0, 0, 1, false, false, true>},
                                         {filter_mma_kernel<2, 0, 0, 0, false, true, true>, filter_mma_kernel<2, 0, 0, 1, false, true, true>}};
    KernelFn fn;
    if (self_mode)    fn = self2[euclid ? 1 : 0][p.grid_updates ? 1 : 0];
    else if (euclid)  fn = euclid2[p.grid_updates ? 1 : 0];
    else if (cg == 2) fn = instr ? instr2[nm] : prod2[nm][(p.grid_exact ? 2 : 0) + (p.grid_updates ? 1 : 0)];
    else              fn = instr ? instr1[nm] : prod1[nm];
    // the opt-in to > 48 KB of dynamic shared memory is a per-DEVICE function attribute: set once per device this process uses
    {
        static std::mutex mu;
        static bool attr_set[kMaxDevices] = {};
        const int slot = current_device_slot();
        std::lock_guard<std::mutex> lock(mu);
        if (!attr_set[slot]) {
            for (int m = 0; m < 4; ++m) {
                for (int v = 0; v < 4; ++v)
                    FFR_CUDA_TRY(cudaFuncSetAttribute(prod2[m][v], cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
                FFR_CUDA_TRY(cudaFuncSetAttribute(instr2[m], cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
                FFR_CUDA_TRY(cudaFuncSetAttribute(prod1[m], cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
                FFR_CUDA_TRY(cudaFuncSetAttribute(instr1[m], cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
            }
            for (int v = 0; v < 2; ++v) {
                FFR_CUDA_TRY(cudaFuncSetAttribute(euclid2[v], cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
                FFR_CUDA_TRY(cudaFuncSetAttribute(self2[0][v], cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
                FFR_CUDA_TRY(cudaFuncSetAttribute(self2[1][v], cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
            }
            attr_set[slot] = true;
        }
    }
    const int64_t n_tiles = (n_cand + kTileM * cg - 1) / (kTileM * cg);
    const int64_t max_groups = sms / cg;
    const unsigned grid = static_cast<unsigned>((n_tiles < max_groups ? n_tiles : max_groups) * cg);
    g_last_cfg[0] = cg; g_last_cfg[1] = p.grid_exact; g_last_cfg[2] = p.grid_updates; g_last_cfg[3] = nm;
    g_last_cfg[4] = a_stages; g_last_cfg[5] = b_stages; g_last_cfg[6] = static_cast<int>(grid); g_last_cfg[7] = instr ? 1 : 0;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(64 + 32 * ew + (fuse ? 64 : 0));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cg; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (after_k1 && n_ref_dev == nullptr) {   // the previous launch of this stream is K1 (it triggers its dependents at entry)
        attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[1].val.programmaticStreamSerializationAllowed = 1;
        cfg.numAttrs = 2;
    }
    FFR_CUDA_TRY(cudaLaunchKernelEx(&cfg, fn, tm_c, tm_r, tm_c32, p));
    FFR_LAUNCH_CHECK("filter_mma");
    return FFR_OK;
}

}  // namespace

// true when ffr_filter skips the K1 pass over the candidates and lets K2's normaliser warps do it behind the MMAs.
// That needs float4-addressable rows and enough tensor work per candidate tile to hide two warps' worth of loads
// (~8 GB/s per SM): with few reference tiles per candidate tile the kernel would wait for its own normaliser, and the
// separate full-bandwidth K1 pass is the better schedule.  FFR_FUSE_K1=0|1 forces the choice (tests).
bool filter_mma_can_fuse(const float* cand32, int64_t n_ref, int64_t n_cand, int32_t dim, int32_t dim_pad) {
    if (cand32 == nullptr || (dim % 4) != 0 || (reinterpret_cast<uintptr_t>(cand32) & 15) != 0) return false;
    const int forced = knobs().fuse_k1;
    if (forced >= 0) return forced != 0;
    // Tensor time per candidate tile ~ n_rt * (dim_pad / 64) * 512 cycles; the two normaliser warps keep <= 16 KB in flight per
    // SM (~7 B/cycle against HBM latency), i.e. ~75 * dim cycles per 128-row tile: hidden with 2x margin from ~20 reference
    // tiles up, whatever the dim.  Few candidate tiles per CTA would expose the first tile's un-hidden pass instead.
    const int64_t n_rt = (n_ref + kTileN - 1) / kTileN;
    // stage32 (128-d rows): the fp32 rows come through a TMA-fed shared-memory ring, two warps convert a tile in ~4 k cycles
    // -- hidden behind even ONE reference tile's epilogue -- so the K1 pass over the candidates goes whatever n_ref is
    if (filter_mma_stage32_ok(dim, dim_pad) && knobs().cta_group == 2)
        return n_cand >= 4 * static_cast<int64_t>(kTileM) * num_sms();
    return n_rt >= 24 && n_cand >= 4 * static_cast<int64_t>(kTileM) * num_sms();
}

int launch_filter_mma(const __half* ref16, int64_t n_ref, __half* cand16, const float* cand32, int32_t dim,
                      int64_t n_cand, int32_t dim_pad,
                      float thr, float delta, float thr_band, int64_t ref_index_base, uint8_t* keep, int32_t* idx, float* val,
                      RecheckLists lists, int no_recheck, float band_tol, int32_t* band_count, int64_t* band_rows,
                      int64_t band_cap, bool after_k1, const int32_t* ref_map, const int32_t* n_ref_dev, cudaStream_t s,
                      const float* euclid_bias, const float* cand_scale, const float* bias_max, SelfArgs self) {
    return launch_filter_mma_impl(ref16, n_ref, cand16, cand32, dim, n_cand, dim_pad, thr, delta, thr_band, ref_index_base,
                                  keep, idx, val, lists, no_recheck, BandArgs{band_tol, band_count, band_rows, band_cap}, nullptr,
                                  after_k1, ref_map, n_ref_dev, s, euclid_bias, cand_scale, bias_max, self);
}

// true when the fused schedule needs NO fp16 copy of the candidates in the workspace (stage32: the fp16 A tiles only ever
// exist in shared memory), decided from the shape alone -- ffr_filter_workspace_bytes sizes the workspace with it.  The
// candidate pointer is assumed 16-byte aligned (the header's contract); a misaligned one is rejected by ffr_filter.
bool filter_mma_skips_cand16(int64_t n_ref, int64_t n_cand, int32_t dim) {
    const int32_t dim_pad = (dim + 63) / 64 * 64;
    const Knobs& kn = knobs();
    if (kn.cta_group != 2 || (num_sms() & 1)) return false;
    if (!filter_mma_stage32_ok(dim, dim_pad)) return false;
    return filter_mma_can_fuse(reinterpret_cast<const float*>(uintptr_t(256)), n_ref, n_cand, dim, dim_pad);
}

void set_mma_prof_buffer(unsigned long long* dev_ptr) { g_prof.store(dev_ptr, std::memory_order_relaxed); }
void get_last_k2_config(int out[8]) { for (int i = 0; i < 8; ++i) out[i] = g_last_cfg[i]; }

// test hook (not part of the ABI in include/ffr.h): additionally dumps the full score matrix
int launch_filter_mma_debug(const __half* ref16, int64_t n_ref, const __half* cand16, int64_t n_cand, int32_t dim_pad,
                            float thr, float delta, uint8_t* keep, int32_t* idx, float* val, RecheckLists lists,
                            float* scores, cudaStream_t s) {
    return launch_filter_mma_impl(ref16, n_ref, const_cast<__half*>(cand16), nullptr, dim_pad, n_cand, dim_pad, thr, delta, delta, 0, keep, idx,
                                  val, lists, 0, BandArgs{0.f, nullptr, nullptr, 0}, scores, false, nullptr, nullptr, s,
                                  nullptr, nullptr, nullptr, kNoSelf);
}

}  // namespace ffr

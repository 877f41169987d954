// Shared helpers for the ffr CUDA sources: error plumbing, launch accounting, sm_100a PTX wrappers.
#pragma once

#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/ffr.h"

namespace ffr {

// ---- host-side error plumbing -------------------------------------------------------------------
void set_error(const char* fmt, ...);
int  cuda_fail(cudaError_t e, const char* what);          // records message, returns FFR_ERR_CUDA
void count_launch(int n = 1);

#define FFR_CUDA_TRY(expr)                                                   \
    do {                                                                     \
        cudaError_t _e = (expr);                                             \
        if (_e != cudaSuccess) return ::ffr::cuda_fail(_e, #expr);           \
    } while (0)

#define FFR_LAUNCH_CHECK(name)                                               \
    do {                                                                     \
        cudaError_t _e = cudaGetLastError();                                 \
        if (_e != cudaSuccess) return ::ffr::cuda_fail(_e, name);            \
        ::ffr::count_launch();                                               \
    } while (0)

int num_sms();                                             // SM count of the current device (cached)
int current_device_slot();                                 // cudaGetDevice clamped to [0, kMaxDevices): index of per-device caches
constexpr int kMaxDevices = 64;

// ---- dispatch overrides (FFR_* environment variables, DESIGN.md §10) ------------------------------------
// Each one forces a choice the dispatcher also makes by itself on some shape or platform (tests use them to reach those
// paths at small sizes).  Read from the environment ONCE per process (first use); the hot path never calls getenv.  Tests
// that flip one between calls use the non-ABI hook ffr_debug_reload_env().  -1 = "auto" where the default depends on the shape.
struct Knobs {
    int cta_group, grid_update_refs, grid_exact, fuse_k1, stage32, dedup_refs, tail_offload;
};
const Knobs& knobs();
void reload_knobs();
float recheck_delta();                                     // K3 window in cosine units (DESIGN.md §4); test hook can change it

// ---- layout of the per-row recheck record K2 -> K3 ------------------------------------------------
struct RecheckRec {     // pair record (K3a)                                  | part record (K3p, written from the END of the array)
    int32_t row;        // candidate row (local)                              | same
    int32_t idx1;       // best reference (local index), fp16-score space     | (first compact column of the span >> 7) | Y-group mask << 24
    int32_t idx2;       // runner-up reference, or -1                         | one tracked candidate outside the span, or -1
    int32_t idx3;       // third reference inside the window, or -1           | X-group mask: 16 bits per 128-column part (one or two adjacent parts)
};

// rows whose third-best score is also within delta: rescanned against every reference in fp32 (K3b).
// K2 appends the row, zeroes its packed-result key and the arrival counter of its group of kFullGroup rows.
constexpr int kFullGroup = 16;
struct WsHeader;
struct RecheckLists {
    WsHeader* hdr;
    RecheckRec* recs;          // near-tie / near-threshold rows: two-candidate fp32 check (K3a) from the front; part-rescan
                               // records {row, first reference of the part, two more candidates} from the back
    int64_t rec_cap;
    int32_t* full_rows;        // rows needing the full rescan (K3b)
    unsigned long long* full_keys;   // per full row: (orderable(best) << 32) | ~idx, combined with atomicMax
    int32_t* full_ctr;         // per group of kFullGroup full rows: blocks that have contributed
    int64_t full_cap;
};

// workspace header shared by all filter paths (device memory, 256 B)
struct WsHeader {
    int32_t recheck_count;   // rows appended to the recheck list
    int32_t full_count;      // of which need the full rescan
    int32_t path;            // 0 fp32, 1 mma
    int32_t launches;
    int32_t part_count;      // rows whose hidden columns all lie in one 128-reference part (records at the END of recs, growing down)
    int32_t refs_scanned;    // reference rows K2 actually scanned (< n_ref when exact duplicates were folded)
    // match lists (ffr_match_pairs*): K2's raw pair list and exact-row list, the finishing pass's counters
    int32_t exact_count;     // Euclid candidates whose scores are unusable (1 / |c| not finite): scanned in fp32
    int32_t pairs_blocks;    // finishing-pass blocks done (the last one writes the caller's count)
    unsigned long long raw_count;      // pairs K2 listed (keeps counting past the raw list's capacity)
    unsigned long long acc_count;      // pairs the finishing pass accepted (slots of the caller's list)
    unsigned long long acc_exact;      // ... of which from the exact-row list
    int32_t pad[50];
};
static_assert(sizeof(WsHeader) == 256, "the workspace header is 256 bytes");

// A match-list call's outputs (ffr_match_pairs*): accepted pairs go to [0, cap), *count is written by the last kernel
struct PairOut {
    int32_t* cand;
    int32_t* ref;
    float* val;
    int64_t cap;
    int64_t* count;
};
// K2's pairs form: raw (candidate row, reference column) entries, exact rows (Euclid candidates with unusable scores)
struct PairRaw {
    uint2* raw;
    int64_t cap;
    int32_t* exact_rows;
    const uint32_t* e_max_bits;   // Euclid: E1's largest squared reference norm (bits), from which K2 derives E2's 2^-f
};

// Self mode (ffr_filter_self): the candidates are rows [row0, row0 + n_cand) of the reference matrix itself, and candidate row g
// (global index) may not match reference i == g (FFR_SELF_OTHERS) or any i >= g (FFR_SELF_EARLIER).  mode < 0: gallery call.
struct SelfArgs {
    int64_t row0;
    int mode;
};
constexpr SelfArgs kNoSelf = {0, -1};

// ---- a filter call's outputs (host launchers; K2s and the value pass take Band as a kernel parameter) ----------------------
// Rows with |best - thr| <= tol are appended (unordered) to rows[0..cap) and counted in *count (which may exceed cap);
// count nullptr: no band.
struct Band {
    float tol;
    int32_t* count;
    int64_t* rows;
    int64_t cap;
};
struct FilterOut {
    uint8_t* keep;
    int32_t* idx;
    float* val;            // may be nullptr
    Band band;
};

// ---- device helpers -------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ bool self_eligible(int64_t i, int64_t g, int mode) {
    return i >= 0 && (mode == FFR_SELF_EARLIER ? i < g : i != g);
}

// ---- programmatic dependent launch (K1 -> K2 -> K3 without launch gaps) ----
// pdl_launch_dependents: the NEXT kernel of the stream (if it was launched with the programmatic-serialisation attribute)
// may start now instead of when this grid has drained.  pdl_wait: blocks until the PREVIOUS grid has completed and its
// writes are visible; a no-op for a kernel launched without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// |c - m|_2 of one row with EXACTLY the per-lane element assignment, accumulation order and reduction tree the streaming
// filter K2s uses for an Euclid score (ffr_filter_fp32.cu), so that K5's threshold -- the largest reference-to-mean distance --
// is bit-identical to the distance the filter later computes for that same reference as a candidate (the reference gets both
// from one np.linalg.norm: the farthest reference always passes `<= thres`, filter_faces_using_reference.py:88-99,189).
// mode (k2s_form on the host): 0 = scalar lane-strided; 1, 2, 4, 8 = float4 #(lane + 32 j), j < mode; 16 / 32 = sub-warp
// form, 8 / 16 lanes per row with float4 #(sub + L j), j < 4.  The whole warp calls it; every lane returns the distance.
__device__ __forceinline__ float k2s_euclid_dist(const float* __restrict__ c, const float* m, int32_t dim, int lane, int mode) {
    float a = 0.f;
    if (mode == 0) {
        for (int k = lane; k < dim; k += 32) { const float d = c[k] - m[k]; a = fmaf(d, d, a); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    } else {
        const float4* c4 = reinterpret_cast<const float4*>(c);
        const float4* m4 = reinterpret_cast<const float4*>(m);
        const int nvec = dim >> 2;
        const int L = mode >= 16 ? mode / 2 : 32, nj = mode >= 16 ? 4 : mode, sub = lane % L;
        for (int j = 0; j < nj; ++j) {
            const int k = sub + L * j;
            if (k < nvec) {
                const float4 cv = c4[k], mv = m4[k];
                float d;
                d = cv.x - mv.x; a = fmaf(d, d, a);
                d = cv.y - mv.y; a = fmaf(d, d, a);
                d = cv.z - mv.z; a = fmaf(d, d, a);
                d = cv.w - mv.w; a = fmaf(d, d, a);
            }
        }
        for (int o = L / 2; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    }
    return __fsqrt_rn(a);
}

// E2's power of two (ffr_l2norm.cu): 2^-f with f the smallest integer such that 2^(2f) > mx = the largest squared reference norm
__device__ __forceinline__ float euclid_ref_scale(float mx) {
    int e = 0;
    if (mx > 0.f && mx <= 3.4e38f) frexpf(mx, &e);                     // mx < 2^e
    const int f = (e + 1) >> 1;                                         // |r| < 2^(e/2) <= 2^f
    return ldexpf(1.0f, -f);
}

__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

// streaming load that also tells L2 to evict the line first (data read exactly once)
__device__ __forceinline__ float4 ldg_stream_evict_first_f4(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(0x12F0000000000000ull));
    return r;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier ----
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_global() {
    asm volatile("fence.proxy.async.global;" ::: "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_shared(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
    return v;
}
__device__ __forceinline__ void red_release_shared_add(uint32_t* p, uint32_t v) {
    asm volatile("red.release.cta.shared::cta.add.u32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// non-blocking probe (try_wait may suspend the thread for a system-dependent time; a loop that watches two barriers
// must not)
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) { }
}

// ---- TMA ----
__device__ __forceinline__ void tma_prefetch_desc(const void* desc) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(desc) : "memory");
}
// 2D tiled load: coordinates (c0 = innermost/K element index, c1 = row index)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* desc, uint64_t* bar,
                                            int32_t c0, int32_t c1, uint64_t cache_hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(desc), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(cache_hint)
        : "memory");
}
constexpr uint64_t kEvictFirst  = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast   = 0x14F0000000000000ull;

// ---- tcgen05 ----
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after()  { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst) {      // whole warp, .sync.aligned
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(smem_dst)), "n"(kCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {        // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]^T, kind::f16 (fp16 operands, fp32 accumulate), one thread issues
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on an mbarrier once all previously issued MMAs of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                 ::"r"(smem_u32(bar)) : "memory");
}

// 32 lanes x 32 columns of fp32: thread l of the warp receives row (lane_base + l), columns col..col+31
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float (&v)[32]) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
// 32 lanes x 64 columns of fp32: thread l receives row (lane_base + l), columns col..col+63
__device__ __forceinline__ void tmem_ld_32x64(uint32_t taddr, float (&v)[64]) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// tcgen05.ld is asynchronous: its destination registers are defined only after tcgen05.wait::ld.  The compiler does not
// know that (consumers only depend on the ld statement) and is free to hoist arithmetic on v above the wait; this empty
// statement, placed after tmem_ld_wait(), redefines v so every use stays below it.  No instruction is emitted.
__device__ __forceinline__ void tmem_ld_fence(float (&v)[32]) {
    asm volatile("" : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]),
                      "+f"(v[8]), "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15]),
                      "+f"(v[16]), "+f"(v[17]), "+f"(v[18]), "+f"(v[19]), "+f"(v[20]), "+f"(v[21]), "+f"(v[22]), "+f"(v[23]),
                      "+f"(v[24]), "+f"(v[25]), "+f"(v[26]), "+f"(v[27]), "+f"(v[28]), "+f"(v[29]), "+f"(v[30]), "+f"(v[31])
                 :: "memory");
}

__device__ __forceinline__ float fmax3(float a, float b, float c) {
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// UMMA shared-memory matrix descriptor, K-major operand, SWIZZLE_128B, rows of 64 fp16 (128 B):
//   start address >> 4 in [0,14); LBO (ignored for swizzled K-major) = 1 in [16,30);
//   SBO = 1024 B (8 rows x 128 B) >> 4 = 64 in [32,46); version 1 in [46,48); layout SWIZZLE_128B = 2 in [61,64).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>(1) << 16;
    d |= static_cast<uint64_t>(1024 >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}

// instruction descriptor, kind::f16: D fp32 (c_format 1 at [4,6)), A/B fp16 (0), both K-major,
// N>>3 at [17,23), M>>4 at [24,29)
__device__ __host__ constexpr uint32_t umma_idesc_f16(uint32_t m, uint32_t n) {
    return (1u << 4) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

#endif  // __CUDACC__

// ---- kernel launchers implemented in the .cu files (host) ----------------------------------------
int launch_l2norm(const float* x, int64_t rows, int32_t dim, __half* y16, int32_t ld16, float* y32, float* norms,
                  cudaStream_t s);
int launch_filter_fp32(const float* ref, int64_t n_ref, const float* cand, int64_t n_cand, int32_t dim, int metric,
                       float thr, int64_t ref_index_base, const FilterOut& out, cudaStream_t s);
// K2s self form: candidates x[self.row0 .. self.row0 + n_cand) against all n rows of x, excluded references skipped
int launch_filter_fp32_self(const float* x, int64_t n, int64_t n_cand, int32_t dim, int metric, SelfArgs self, float thr,
                            const FilterOut& out, cudaStream_t s);
// The form K2s scores (ref, cand) row pairs with when it scans n_ref references (launch_filter_fp32 dispatches on it):
// 0 = scalar lane-strided; 1, 2, 4, 8 = float4 per lane; 16 / 32 = the sub-warp kernel (n_ref <= 2, dim 128 / 256).  Every
// kernel whose Euclid distance must be K2s's bit for bit (K5, K3's Euclid form, the value pass, the all-reduce merge) takes
// k2s_euclid_dist's mode from it.
int k2s_form(const float* ref, const float* cand, int64_t n_ref, int32_t dim);
int launch_l2norm_pair(const float* x_a, int64_t rows_a, __half* y16_a, const float* x_b, int64_t rows_b, __half* y16_b,
                       int32_t dim, int32_t ld16, void* zero_ptr, int32_t zero_words, cudaStream_t s,
                       float* scale_a = nullptr);
// Euclid on the tensor cores (ffr_l2norm.cu): fp16(r * 2^-f) rows, f from the largest reference norm (device side), and the
// per-reference bias beta_i = -|r_i|^2 * 2^-f / 2 (zero padded to a multiple of 256); bmax[0] = max_i |beta_i|.
// nsq: n_ref floats of scratch, max_bits: one zeroed-here word.
int launch_euclid_refs(const float* ref, int64_t n_ref, int32_t dim, int32_t ld16, __half* ref16, float* beta, float* nsq,
                       uint32_t* max_bits, float* bmax, cudaStream_t s);
inline int64_t euclid_bias_len(int64_t n_ref) { return (n_ref + 255) / 256 * 256; }
bool filter_mma_can_fuse(const float* cand32, int64_t n_ref, int64_t n_cand, int32_t dim, int32_t dim_pad);
int launch_filter_mma(const __half* ref16, int64_t n_ref, __half* cand16, const float* cand32, int32_t dim,
                      int64_t n_cand, int32_t dim_pad, float thr, float delta, float thr_band, int64_t ref_index_base,
                      const FilterOut& out, RecheckLists lists, int no_recheck, bool after_k1, const int32_t* ref_map,
                      const int32_t* n_ref_dev, cudaStream_t s,
                      const float* euclid_bias = nullptr, const float* cand_scale = nullptr, const float* bias_max = nullptr,
                      SelfArgs self = kNoSelf, const PairRaw* pairs = nullptr);
// Match lists (ffr_recheck.cu).  Finishing pass behind K2's pairs form: the fp32 value of every raw entry (and of every exact row
// against every reference), accepted pairs appended to out, *out.count written by the last block.  self.mode >= 0: cand is rows
// [self.row0, ...) of ref (references i < g only).
int launch_pairs_finish(const float* ref, int64_t n_ref, const float* cand, int32_t dim, int metric, float thr, int64_t ref_index_base,
                        SelfArgs self, const PairRaw& raw, WsHeader* hdr, const PairOut& out, cudaStream_t s);
// The exact path: one warp per candidate row over every reference, the same value arithmetic; *out.count must be zero before
int launch_pairs_exact(const float* ref, int64_t n_ref, const float* cand, int64_t n_cand, int32_t dim, int metric, float thr,
                       int64_t ref_index_base, SelfArgs self, const PairOut& out, cudaStream_t s);
// Near-duplicate groups (ffr_groups.cu): labels[i] = i and *group_count = 0; then the union-find over the edges (edge_a[k],
// edge_b[k]), k < min(*filled, cap) (*filled read on the device), and the final labels (each row's smallest component row) with
// their count
int launch_groups_init(int32_t* labels, int64_t n, int64_t* group_count, cudaStream_t s);
int launch_groups_union(const int32_t* edge_a, const int32_t* edge_b, int64_t cap, const unsigned long long* filled, int32_t* labels,
                        int64_t n, int64_t* group_count, cudaStream_t s);
// exact-duplicate reference rows folded before K2 (ffr_dedup.cu)
bool dedup_wanted(int64_t n_ref, int64_t n_cand);
size_t dedup_workspace_bytes(int64_t n_ref, int32_t ld);
int launch_dedup_refs(const float* ref32, const __half* ref16_full, int64_t n_ref, int32_t dim, int32_t ld, void* ws,
                      __half** out_ref16, int32_t** out_map, int32_t** out_n_unique_dev, cudaStream_t s,
                      const float* bias = nullptr, float* bias_c = nullptr);   // Euclid: the bias is compacted with the rows
bool filter_mma_skips_cand16(int64_t n_ref, int64_t n_cand, int32_t dim);
void get_last_k2_config(int out[8]);
int launch_recheck(const float* ref, int64_t n_ref, const float* cand, int64_t n_cand, int32_t dim, float thr,
                   int64_t ref_index_base, const FilterOut& out, RecheckLists lists, const int32_t* ref_map,
                   const int32_t* n_unique_dev, cudaStream_t s, int euclid_mode = -1, SelfArgs self = kNoSelf);
// Euclid after the tensor-core pass: keep / best_val / band from the K2s distance to the chosen reference out.idx (only read)
// (ffr_filter_fp32.cu)
int launch_euclid_values(const float* ref, const float* cand, int64_t n_cand, int32_t dim, float thr, int64_t ref_index_base,
                         const FilterOut& out, int mode, cudaStream_t s, bool self = false);
int launch_ref_stats_batched(const float* ref_feat, const int32_t* offsets, int32_t n_classes, int32_t dim, float* mean,
                             float* thres, cudaStream_t s);
int launch_first_match_stream(float* g_feat, float* g_bbox, int32_t* g_count, int32_t cap, const float* queries,
                              const float* qboxes, int32_t n_queries, int32_t dim, int metric, float normal_thres,
                              float harsh_thres, int32_t* match_idx, cudaStream_t s);
void set_mma_prof_buffer(unsigned long long* dev_ptr);   // diagnostics: [grid][16] stall-cycle counters of K2
int launch_ref_stats(const float* ref_feat, int32_t n_ref, int32_t dim, float* mean, float* thres, cudaStream_t s);
// gallery over ranks (ffr_recheck.cu): the merge key of each row's winner on this rank, and the outputs from the reduced keys
int launch_best_keys(const float* ref, int64_t n_ref, int64_t ref_index_base, const float* cand, int64_t n_cand, int32_t dim,
                     int metric, const int32_t* best_idx, unsigned long long* keys, cudaStream_t s);
int launch_emit_keys(const unsigned long long* keys, int64_t n_cand, int metric, float thr, const FilterOut& out, cudaStream_t s);
int launch_pack_results(const uint8_t* keep, const int32_t* idx, int64_t m, int64_t m_pad, uint8_t* packed,
                        cudaStream_t s);
int launch_unpack_results(const uint8_t* packed, int64_t m, int64_t m_pad, int nranks, uint8_t* keep, int32_t* idx,
                          cudaStream_t s);
int launch_filter_mma_debug(const __half* ref16, int64_t n_ref, const __half* cand16, int64_t n_cand, int32_t dim_pad,
                            float thr, float delta, const FilterOut& out, RecheckLists lists, float* scores, cudaStream_t s);

}  // namespace ffr

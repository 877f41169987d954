// C-ABI entry points of libffr_b200.so (declared in include/ffr.h): argument checking, dispatch between
// the exact fp32 CUDA-core kernel and the tcgen05 kernel, workspace carving, the host-buffer pipeline
// (ffr_ctx_*), the NCCL gather (ffr_comm_*, NCCL dlopen'ed so the library loads without it) and the merge of a gallery
// sharded over ranks (ffr_allreduce_best).
#include <dlfcn.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <new>

#include "ffr_common.cuh"

#define FFR_STR2(x) #x
#define FFR_STR(x) FFR_STR2(x)

namespace ffr {

namespace {
thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};
std::atomic<float> g_delta{4e-4f};       // recheck window in cosine units, see DESIGN.md §4 (fp16 operand rounding)
std::atomic<const Knobs*> g_knobs{nullptr};
std::mutex g_knobs_mu;
struct LastCall { const void* ws; int path; int launches; };
thread_local LastCall g_last = {nullptr, 0, 0};
// profiling hook: CUDA events recorded on the launch stream right before / after the tcgen05 kernel
thread_local cudaEvent_t g_ev_k2_begin = nullptr, g_ev_k2_end = nullptr;
}  // namespace

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) at %s", static_cast<int>(e), cudaGetErrorString(e), what);
    return FFR_ERR_CUDA;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int current_device_slot() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) return 0;
    return dev < kMaxDevices ? dev : kMaxDevices - 1;
}

int num_sms() {
    static std::atomic<int> cached[kMaxDevices];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return 148;
    int n = cached[dev].load(std::memory_order_relaxed);
    if (n == 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev].store(n, std::memory_order_relaxed);
    }
    return n;
}

namespace {
int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v != nullptr && *v) ? atoi(v) : dflt;
}
const Knobs* read_knobs() {
    Knobs* k = new Knobs();
    k->cta_group = env_int("FFR_CTA_GROUP", 2);
    k->grid_update_refs = env_int("FFR_GRID_UPDATE_REFS", 8192);
    k->grid_exact = env_int("FFR_GRID_EXACT", -1);
    k->fuse_k1 = env_int("FFR_FUSE_K1", -1);
    k->stage32 = env_int("FFR_STAGE32", 1);
    k->dedup_refs = env_int("FFR_DEDUP_REFS", 1);
    k->tail_offload = env_int("FFR_TAIL_OFFLOAD", -1);
    return k;
}
}  // namespace

const Knobs& knobs() {
    const Knobs* k = g_knobs.load(std::memory_order_acquire);
    if (k == nullptr) {
        std::lock_guard<std::mutex> lock(g_knobs_mu);
        k = g_knobs.load(std::memory_order_acquire);
        if (k == nullptr) { k = read_knobs(); g_knobs.store(k, std::memory_order_release); }
    }
    return *k;
}
// test hook: the previous snapshot is leaked on purpose (another thread may still hold a reference to it)
void reload_knobs() {
    std::lock_guard<std::mutex> lock(g_knobs_mu);
    g_knobs.store(read_knobs(), std::memory_order_release);
}
float recheck_delta() { return g_delta.load(std::memory_order_relaxed); }

namespace {

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct WsLayout {
    size_t hdr, ref16, cand16, recs, full_rows, full_keys, full_ctr, dedup, total;
    size_t e_bias, e_bias_c, e_nsq, e_scal, e_cscale;     // Euclid on the tensor cores (see EuclidWs)
    bool mma;
};

// The tcgen05 Euclid kernel exists for cta_group::2 only (an SM count that pairs up, FFR_CTA_GROUP=2): elsewhere Euclid keeps the
// exact CUDA-core kernel K2s, like every other shape the tensor-core path does not take.
bool euclid_mma_available() { return knobs().cta_group == 2 && (num_sms() & 1) == 0; }

bool mma_eligible(int64_t n_ref, int32_t dim, int metric, int flags) {
    if (metric == FFR_METRIC_EUCLID)   // K3 always re-checks Euclid: without it (FFR_FLAG_NO_RECHECK) the exact K2s path runs
        return !(flags & FFR_FLAG_FORCE_FP32) && dim <= 512 && n_ref > 8 && !(flags & FFR_FLAG_NO_RECHECK) &&
               euclid_mma_available();
    if (metric != FFR_METRIC_COSINE) return false;
    if (flags & FFR_FLAG_FORCE_FP32) return false;
    if (dim > 512) return false;
    if (flags & FFR_FLAG_FORCE_MMA) return true;
    return n_ref > 8;          // <= 8 references: the streaming fp32 kernel is already HBM-bound and exact
}

// need_c16: the fp16 copy of the candidates lives in the workspace (false for fp16 input and for stage32, whose fp16 A
// tiles only ever exist in shared memory: 320 MB less at BASELINE configs[4]'s shard)
// euclid: the tcgen05 Euclid path's extra buffers -- the reference bias (and its deduplicated copy), the references' squared
// norms, two scalars, and the candidates' 1 / |c| (n_ref == 0: the caller prepared the references)
WsLayout ws_layout(int64_t n_ref, int64_t n_cand, int32_t dim, int dtype, bool mma, bool need_c16, bool dedup,
                   bool euclid = false) {
    WsLayout L{};
    L.mma = mma;
    size_t off = 0;
    L.hdr = off; off += align_up(sizeof(WsHeader), 256);
    if (mma) {
        const size_t ld = static_cast<size_t>(ffr_padded_dim(dim));
        L.ref16 = off;  if (dtype == FFR_DTYPE_F32) off += align_up(static_cast<size_t>(n_ref) * ld * 2, 256);
        L.cand16 = off; if (dtype == FFR_DTYPE_F32 && need_c16) off += align_up(static_cast<size_t>(n_cand) * ld * 2, 256);
        L.recs = off;      off += align_up(static_cast<size_t>(n_cand) * sizeof(RecheckRec), 256);
        L.full_rows = off; off += align_up(static_cast<size_t>(n_cand) * sizeof(int32_t), 256);
        L.full_keys = off; off += align_up(static_cast<size_t>(n_cand) * sizeof(unsigned long long), 256);
        L.full_ctr = off;  off += align_up((static_cast<size_t>(n_cand) / kFullGroup + 1) * sizeof(int32_t), 256);
        L.dedup = off;     if (dedup && dtype == FFR_DTYPE_F32) off += align_up(dedup_workspace_bytes(n_ref, static_cast<int32_t>(ld)), 256);
        if (euclid) {
            const size_t nb = n_ref > 0 ? static_cast<size_t>(euclid_bias_len(n_ref)) * 4 : 0;
            L.e_bias = off;    off += align_up(nb, 256);
            L.e_bias_c = off;  if (dedup) off += align_up(nb, 256);
            L.e_nsq = off;     off += align_up(static_cast<size_t>(n_ref) * 4, 256);
            L.e_scal = off;    off += 256;
            L.e_cscale = off;  off += align_up(static_cast<size_t>(n_cand) * 4, 256);
        }
    }
    L.total = off;
    return L;
}

int check_common(const void* ref, int64_t n_ref, const void* cand, int64_t n_cand, int32_t dim, int dtype, int metric,
                 const uint8_t* keep, const int32_t* idx) {
    if (n_ref <= 0) { set_error("n_ref must be > 0 (got %lld)", (long long)n_ref); return FFR_ERR_INVALID; }
    if (n_cand < 0) { set_error("n_cand must be >= 0 (got %lld)", (long long)n_cand); return FFR_ERR_INVALID; }
    if (dim <= 0) { set_error("dim must be > 0 (got %d)", dim); return FFR_ERR_INVALID; }
    if (ref == nullptr || (n_cand > 0 && (cand == nullptr || keep == nullptr || idx == nullptr))) {
        set_error("null pointer argument");
        return FFR_ERR_INVALID;
    }
    if (dtype != FFR_DTYPE_F32 && dtype != FFR_DTYPE_F16) { set_error("unknown dtype %d", dtype); return FFR_ERR_INVALID; }
    if (metric != FFR_METRIC_COSINE && metric != FFR_METRIC_EUCLID) { set_error("unknown metric %d", metric); return FFR_ERR_INVALID; }
    return FFR_OK;
}

// core: ref16_pre != nullptr -> references already normalised/converted (ctx pipeline caches them)
// ref16_pre != nullptr: the caller already holds the prepared references (fp16, normalised; when map_pre / nuniq_pre are given:
// exact duplicates folded, see ffr_dedup.cu)
// ref16_pre with metric Euclid: fp16(r * 2^-f) rows, and euclid_pre = {bias, bias_max} (launch_euclid_refs)
int filter_core(const void* ref, const __half* ref16_pre, const int32_t* map_pre, const int32_t* nuniq_pre, int64_t n_ref,
                const void* cand, int64_t n_cand, int32_t dim,
                int dtype, int metric, float thr, int64_t ref_index_base, uint8_t* keep, int32_t* best_idx,
                float* best_val, float band_tol, int32_t* band_count, int64_t* band_rows, int64_t band_cap, int flags,
                void* workspace, size_t ws_bytes, cudaStream_t s, const float* const* euclid_pre = nullptr) {
    const bool mma = mma_eligible(n_ref, dim, metric, flags);
    if ((flags & FFR_FLAG_FORCE_MMA) && !mma) {
        set_error("FFR_FLAG_FORCE_MMA: tcgen05 path needs dim <= 512, metric cosine, or metric euclid with n_ref > 8, the re-check "
                  "and cta_group::2 (dim=%d metric=%d n_ref=%lld)", dim, metric, (long long)n_ref);
        return FFR_ERR_UNSUPPORTED;
    }
    const bool euclid = metric == FFR_METRIC_EUCLID;
    if (euclid && dtype != FFR_DTYPE_F32) {
        set_error("metric euclid needs fp32 rows (FFR_DTYPE_F16 rows are normalised: their distances are not the embeddings')");
        return FFR_ERR_UNSUPPORTED;
    }
    const int32_t ld = ffr_padded_dim(dim);
    // K2 normalises the candidates itself (K1 fused) when the shape pays for it; in its stage32 form no fp16 copy exists.
    // (Euclid always takes the K1 schedule: K1 also writes the candidates' 1 / |c|.)
    const bool fuse = mma && !euclid && dtype == FFR_DTYPE_F32 && n_cand > 0 &&
                      filter_mma_can_fuse(static_cast<const float*>(cand), n_ref, n_cand, dim, ld);
    const bool need_c16 = !(fuse && filter_mma_skips_cand16(n_ref, n_cand, dim));
    const bool dedup = mma && dtype == FFR_DTYPE_F32 && ref16_pre == nullptr && dedup_wanted(n_ref, n_cand);
    const WsLayout L = ws_layout(ref16_pre ? 0 : n_ref, n_cand, dim, dtype, mma, need_c16, dedup, mma && euclid);
    if (workspace == nullptr || ws_bytes < L.total) {
        set_error("workspace too small: need %zu bytes, got %zu%s", L.total, workspace ? ws_bytes : (size_t)0,
                  (mma && dtype == FFR_DTYPE_F32 && need_c16 && (reinterpret_cast<uintptr_t>(cand) & 15) != 0)
                      ? " (candidate rows are not 16-byte aligned: the fused schedule ffr_filter_workspace_bytes sized for cannot run)" : "");
        return FFR_ERR_WORKSPACE;
    }
    if (reinterpret_cast<uintptr_t>(workspace) & 255) { set_error("workspace must be 256-byte aligned"); return FFR_ERR_INVALID; }
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    WsHeader* hdr = reinterpret_cast<WsHeader*>(ws + L.hdr);
    g_last = {workspace, mma ? 1 : 0, 0};
    if (band_count != nullptr) FFR_CUDA_TRY(cudaMemsetAsync(band_count, 0, sizeof(int32_t), s));
    // the re-check header (list counters) must be zero before K2: the K1 launch does it when there is one
    const bool k1_runs = mma && dtype == FFR_DTYPE_F32 && n_cand > 0;
    if (!k1_runs) FFR_CUDA_TRY(cudaMemsetAsync(hdr, 0, sizeof(WsHeader), s));
    if (n_cand == 0) return FFR_OK;

    if (!mma) {
        if (dtype != FFR_DTYPE_F32) {
            set_error("fp16 inputs are only accepted by the tcgen05 cosine path (n_ref > 8, dim <= 512; not with metric euclid)");
            return FFR_ERR_UNSUPPORTED;
        }
        g_last.launches = 1;
        return launch_filter_fp32(static_cast<const float*>(ref), n_ref, static_cast<const float*>(cand), n_cand, dim,
                                  metric, thr, ref_index_base, keep, best_idx, best_val, band_tol, band_count,
                                  band_rows, band_cap, s);
    }

    const __half* ref16 = ref16_pre;
    __half* cand16 = nullptr;
    const float* fuse_cand = nullptr;        // non-null: K2 normalises the candidates itself (K1 fused)
    int launches = 0;
    int rc;
    // Euclid: the reference bias, its maximum and the candidates' 1 / |c| (K2's score is acc + bias * scale)
    const float* e_bias = nullptr;
    const float* e_bmax = nullptr;
    float* e_cscale = nullptr;
    if (mma && euclid) {
        e_cscale = reinterpret_cast<float*>(ws + L.e_cscale);
        if (ref16_pre != nullptr) {
            e_bias = euclid_pre[0]; e_bmax = euclid_pre[1];
        } else {
            __half* r16 = reinterpret_cast<__half*>(ws + L.ref16);
            float* bias = reinterpret_cast<float*>(ws + L.e_bias);
            float* scal = reinterpret_cast<float*>(ws + L.e_scal);
            rc = launch_euclid_refs(static_cast<const float*>(ref), n_ref, dim, ld, r16, bias, reinterpret_cast<float*>(ws + L.e_nsq),
                                    reinterpret_cast<uint32_t*>(scal), scal + 1, s);
            if (rc != FFR_OK) return rc;
            launches += 2;
            ref16 = r16; e_bias = bias; e_bmax = scal + 1;
        }
    }
    if (dtype == FFR_DTYPE_F32) {
        // K1: references (unless the caller cached them) and candidates in ONE launch, which also zeroes the header
        static_assert(sizeof(WsHeader) % 4 == 0 && sizeof(WsHeader) / 4 <= 256, "header is zeroed by one CTA");
        __half* r16 = ref16 == nullptr ? reinterpret_cast<__half*>(ws + L.ref16) : nullptr;
        fuse_cand = fuse ? static_cast<const float*>(cand) : nullptr;
        __half* c16 = need_c16 ? reinterpret_cast<__half*>(ws + L.cand16) : nullptr;
        const bool k1_cand = fuse_cand == nullptr;          // otherwise K2's normaliser warps produce the fp16 rows themselves
        const float* r32 = r16 && !euclid ? static_cast<const float*>(ref) : nullptr;   // (Euclid: prepared above)
        const int64_t r_rows = r32 ? n_ref : 0;
        if (k1_cand) rc = launch_l2norm_pair(static_cast<const float*>(cand), n_cand, c16, r32, r_rows, r16, dim, ld, hdr,
                                             static_cast<int32_t>(sizeof(WsHeader) / 4), s, e_cscale);
        else         rc = launch_l2norm_pair(r32, r_rows, r16, nullptr, 0, nullptr, dim, ld, hdr,
                                             static_cast<int32_t>(sizeof(WsHeader) / 4), s);
        if (rc != FFR_OK) return rc;
        ++launches;
        if (r16 != nullptr) ref16 = r16;
        cand16 = c16;
        if (dedup) {                       // fold bit-identical reference rows: K2 scans the unique ones and maps its columns back
            __half* r16c = nullptr;
            int32_t *map = nullptr, *nuniq = nullptr;
            float* bias_c = euclid ? reinterpret_cast<float*>(ws + L.e_bias_c) : nullptr;
            rc = launch_dedup_refs(static_cast<const float*>(ref), ref16, n_ref, dim, ld, ws + L.dedup, &r16c, &map, &nuniq, s,
                                   euclid ? e_bias : nullptr, bias_c);
            if (rc != FFR_OK) return rc;
            launches += 4;
            ref16 = r16c; map_pre = map; nuniq_pre = nuniq;
            if (euclid) e_bias = bias_c;
        }
    } else {
        if (ref16 == nullptr) ref16 = static_cast<const __half*>(ref);
        cand16 = const_cast<__half*>(static_cast<const __half*>(cand));      // fp16 input: only read
    }
    const bool recheck = (dtype == FFR_DTYPE_F32) && !(flags & FFR_FLAG_NO_RECHECK);
    g_last.launches = launches + 1 + (recheck ? 1 : 0) + (euclid ? 1 : 0);
    RecheckLists lists;
    lists.hdr = hdr;
    lists.recs = reinterpret_cast<RecheckRec*>(ws + L.recs);
    lists.rec_cap = n_cand;
    lists.full_rows = reinterpret_cast<int32_t*>(ws + L.full_rows);
    lists.full_keys = reinterpret_cast<unsigned long long*>(ws + L.full_keys);
    lists.full_ctr = reinterpret_cast<int32_t*>(ws + L.full_ctr);
    lists.full_cap = n_cand;
    const float delta = recheck_delta();
    float thr_band = delta;
    if (band_count != nullptr && band_tol + delta > thr_band) thr_band = band_tol + delta;
    if (g_ev_k2_begin != nullptr) FFR_CUDA_TRY(cudaEventRecord(g_ev_k2_begin, s));
    // Euclid: K2 and K3 only choose the index -- a threshold that never flags a row, no band -- and the value pass decides
    rc = launch_filter_mma(ref16, n_ref, cand16, fuse_cand, dim, n_cand, ld, euclid ? -INFINITY : thr, delta, euclid ? 0.f : thr_band,
                           ref_index_base, keep, best_idx, best_val, lists, recheck ? 0 : 1, band_tol, band_count, band_rows,
                           band_cap, /*after_k1=*/dtype == FFR_DTYPE_F32 && !dedup, map_pre, nuniq_pre, s,
                           e_bias, e_cscale, e_bmax);
    if (rc != FFR_OK) return rc;
    if (g_ev_k2_end != nullptr) FFR_CUDA_TRY(cudaEventRecord(g_ev_k2_end, s));
    const int emode = euclid ? k2s_dist_mode_gallery(static_cast<const float*>(ref), static_cast<const float*>(cand), dim) : -1;
    if (recheck) {
        rc = launch_recheck(static_cast<const float*>(ref), n_ref, static_cast<const float*>(cand), n_cand, dim, nullptr,
                            nullptr, thr, ref_index_base, keep, best_idx, best_val, lists, band_tol,
                            euclid ? nullptr : band_count, band_rows, band_cap, map_pre, nuniq_pre, s, emode);
        if (rc != FFR_OK) return rc;
    }
    if (euclid)
        return launch_euclid_values(static_cast<const float*>(ref), static_cast<const float*>(cand), n_cand, dim, thr,
                                    ref_index_base, keep, best_idx, best_val, band_tol, band_count, band_rows, band_cap, emode, s);
    return FFR_OK;
}

// Self mode (ffr_filter_self): x is both matrices.  K1 normalises x ONCE and, for cosine, the A operand is the candidates' slice
// of that same fp16 copy (kNormMode 0: stage32 or the fused scratch would only read or write those rows a second time).  Euclid
// keeps its operands: E1/E2 turn all n rows into the B operand and its bias, K1 over the slice writes the normalised A rows and
// 1 / |c|.  No duplicate fold: bit-identical rows are what the caller looks for.
bool self_mma_eligible(int64_t n, int32_t dim, int flags) {
    return !(flags & FFR_FLAG_FORCE_FP32) && dim <= 512 && n > 8 && euclid_mma_available();
}

WsLayout self_ws_layout(int64_t n, int64_t n_rows, int32_t dim, int metric, bool mma) {
    const bool euclid = metric == FFR_METRIC_EUCLID;
    return ws_layout(n, n_rows, dim, FFR_DTYPE_F32, mma, /*need_c16=*/euclid, /*dedup=*/false, mma && euclid);
}

int self_core(const float* x, int64_t n, int64_t row_begin, int64_t n_rows, int32_t dim, int metric, int mode, float thr,
              uint8_t* keep, int32_t* best_idx, float* best_val, float band_tol, int32_t* band_count, int64_t* band_rows,
              int64_t band_cap, int flags, void* workspace, size_t ws_bytes, cudaStream_t s) {
    const bool mma = self_mma_eligible(n, dim, flags);
    if ((flags & FFR_FLAG_FORCE_MMA) && !mma) {
        set_error("FFR_FLAG_FORCE_MMA: the self-mode tcgen05 path needs n > 8, dim <= 512 and cta_group::2 (n=%lld dim=%d)",
                  (long long)n, dim);
        return FFR_ERR_UNSUPPORTED;
    }
    const bool euclid = metric == FFR_METRIC_EUCLID;
    const WsLayout L = self_ws_layout(n, n_rows, dim, metric, mma);
    if (workspace == nullptr || ws_bytes < L.total) {
        set_error("workspace too small: need %zu bytes, got %zu", L.total, workspace ? ws_bytes : (size_t)0);
        return FFR_ERR_WORKSPACE;
    }
    if (reinterpret_cast<uintptr_t>(workspace) & 255) { set_error("workspace must be 256-byte aligned"); return FFR_ERR_INVALID; }
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    WsHeader* hdr = reinterpret_cast<WsHeader*>(ws + L.hdr);
    g_last = {workspace, mma ? 1 : 0, 0};
    if (band_count != nullptr) FFR_CUDA_TRY(cudaMemsetAsync(band_count, 0, sizeof(int32_t), s));
    if (!(mma && n_rows > 0)) FFR_CUDA_TRY(cudaMemsetAsync(hdr, 0, sizeof(WsHeader), s));     // (otherwise K1 zeroes it)
    if (n_rows == 0) return FFR_OK;
    const SelfArgs self{row_begin, mode};
    if (!mma) {
        g_last.launches = 1;
        return launch_filter_fp32_self(x, n, n_rows, dim, metric, self, thr, keep, best_idx, best_val, band_tol, band_count,
                                       band_rows, band_cap, s);
    }
    const int32_t ld = ffr_padded_dim(dim);
    const float* cand = x + row_begin * dim;
    __half* x16 = reinterpret_cast<__half*>(ws + L.ref16);
    __half* c16 = nullptr;
    const float *e_bias = nullptr, *e_bmax = nullptr;
    float* e_cscale = nullptr;
    int rc, launches = 0;
    const int32_t hdr_words = static_cast<int32_t>(sizeof(WsHeader) / 4);
    if (euclid) {
        float* bias = reinterpret_cast<float*>(ws + L.e_bias);
        float* scal = reinterpret_cast<float*>(ws + L.e_scal);
        rc = launch_euclid_refs(x, n, dim, ld, x16, bias, reinterpret_cast<float*>(ws + L.e_nsq), reinterpret_cast<uint32_t*>(scal),
                                scal + 1, s);
        if (rc != FFR_OK) return rc;
        c16 = reinterpret_cast<__half*>(ws + L.cand16);
        e_cscale = reinterpret_cast<float*>(ws + L.e_cscale);
        rc = launch_l2norm_pair(cand, n_rows, c16, nullptr, 0, nullptr, dim, ld, hdr, hdr_words, s, e_cscale);
        if (rc != FFR_OK) return rc;
        launches += 3;
        e_bias = bias; e_bmax = scal + 1;
    } else {
        rc = launch_l2norm_pair(x, n, x16, nullptr, 0, nullptr, dim, ld, hdr, hdr_words, s);
        if (rc != FFR_OK) return rc;
        ++launches;
        c16 = x16 + row_begin * ld;
    }
    g_last.launches = launches + 2 + (euclid ? 1 : 0);
    RecheckLists lists;
    lists.hdr = hdr;
    lists.recs = reinterpret_cast<RecheckRec*>(ws + L.recs);
    lists.rec_cap = n_rows;
    lists.full_rows = reinterpret_cast<int32_t*>(ws + L.full_rows);
    lists.full_keys = reinterpret_cast<unsigned long long*>(ws + L.full_keys);
    lists.full_ctr = reinterpret_cast<int32_t*>(ws + L.full_ctr);
    lists.full_cap = n_rows;
    const float delta = recheck_delta();
    float thr_band = delta;
    if (band_count != nullptr && band_tol + delta > thr_band) thr_band = band_tol + delta;
    if (g_ev_k2_begin != nullptr) FFR_CUDA_TRY(cudaEventRecord(g_ev_k2_begin, s));
    rc = launch_filter_mma(x16, n, c16, nullptr, dim, n_rows, ld, euclid ? -INFINITY : thr, delta, euclid ? 0.f : thr_band, 0,
                           keep, best_idx, best_val, lists, 0, band_tol, nullptr, band_rows, band_cap, /*after_k1=*/true,
                           nullptr, nullptr, s, e_bias, e_cscale, e_bmax, self);
    if (rc != FFR_OK) return rc;
    if (g_ev_k2_end != nullptr) FFR_CUDA_TRY(cudaEventRecord(g_ev_k2_end, s));
    const int emode = euclid ? k2s_dist_mode_gallery(x, cand, dim) : -1;
    rc = launch_recheck(x, n, cand, n_rows, dim, nullptr, nullptr, thr, 0, keep, best_idx, best_val, lists, band_tol,
                        euclid ? nullptr : band_count, band_rows, band_cap, nullptr, nullptr, s, emode, self);
    if (rc != FFR_OK) return rc;
    if (euclid)
        return launch_euclid_values(x, cand, n_rows, dim, thr, 0, keep, best_idx, best_val, band_tol, band_count, band_rows,
                                    band_cap, emode, s, /*self=*/true);
    return FFR_OK;
}

}  // namespace
}  // namespace ffr

using namespace ffr;

// ---------------------------------------------------------------------------------------------------
extern "C" {

int ffr_abi_version(void) { return FFR_ABI_VERSION; }
const char* ffr_last_error(void) { return g_err; }
const char* ffr_build_info(void) {
    return "libffr_b200: sm_100a (tcgen05/TMEM/TMA), CUDA " FFR_STR(CUDART_VERSION) ", built " __DATE__;
}
int ffr_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
int32_t ffr_padded_dim(int32_t dim) { return (dim + 63) / 64 * 64; }
int64_t ffr_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

// not in the public header: tuning / test hooks
void ffr_set_recheck_delta(float d) { g_delta.store(d, std::memory_order_relaxed); }
// re-read the FFR_* environment knobs (they are otherwise read once per process)
void ffr_debug_reload_env(void) { reload_knobs(); }
// device buffer [grid][16] u64 that the tcgen05 kernel fills with stall-cycle counters (NULL to disable)
void ffr_debug_set_prof(void* dev_ptr) { set_mma_prof_buffer(static_cast<unsigned long long*>(dev_ptr)); }
// cudaEvent_t pair recorded around the next tcgen05 kernel launches of this thread (NULL, NULL to disable)
void ffr_debug_set_k2_events(void* begin, void* end) {
    g_ev_k2_begin = static_cast<cudaEvent_t>(begin);
    g_ev_k2_end = static_cast<cudaEvent_t>(end);
}
float ffr_get_recheck_delta(void) { return recheck_delta(); }
// {cta_group, grid_exact, grid_updates, normalisation mode (0 K1, 1 fused + scratch, 2 stage32), a_stages, b_stages, grid, instrumented}
// of this thread's last tcgen05 launch
void ffr_debug_last_k2_config(int32_t out[8]) { int v[8]; get_last_k2_config(v); for (int i = 0; i < 8; ++i) out[i] = v[i]; }

int ffr_l2norm_rows_f32(const float* x, int64_t rows, int32_t dim, void* y_f16, int32_t y_f16_ld, float* y_f32,
                        float* norms, ffr_stream_t stream) {
    if (rows < 0 || dim <= 0) { set_error("l2norm: rows >= 0 and dim > 0 required"); return FFR_ERR_INVALID; }
    if (rows == 0) return FFR_OK;
    if (x == nullptr) { set_error("l2norm: x is null"); return FFR_ERR_INVALID; }
    if (y_f16 != nullptr && y_f16_ld < dim) { set_error("l2norm: y_f16_ld %d < dim %d", y_f16_ld, dim); return FFR_ERR_INVALID; }
    if (ffr_device_count() == 0) { set_error("no CUDA device"); return FFR_ERR_CUDA; }
    return launch_l2norm(x, rows, dim, static_cast<__half*>(y_f16), y_f16_ld, y_f32, norms, static_cast<cudaStream_t>(stream));
}

size_t ffr_filter_workspace_bytes(int64_t n_ref, int64_t n_cand, int32_t dim, int dtype, int metric) {
    if (n_ref <= 0 || n_cand < 0 || dim <= 0) return 0;
    // sized for the tcgen05 path whenever it could be chosen (including FFR_FLAG_FORCE_MMA)
    if (metric == FFR_METRIC_EUCLID) {      // the tcgen05 Euclid path (K1 schedule: the fp16 candidates live in the workspace)
        const bool mma = dim <= 512 && n_ref > 8 && dtype == FFR_DTYPE_F32;
        return ws_layout(n_ref, n_cand, dim, dtype, mma, true, mma && dedup_wanted(n_ref, n_cand), mma).total;
    }
    const bool mma = metric == FFR_METRIC_COSINE && dim <= 512;
    const bool need_c16 = !(mma && dtype == FFR_DTYPE_F32 && filter_mma_skips_cand16(n_ref, n_cand, dim));
    return ws_layout(n_ref, n_cand, dim, dtype, mma, need_c16, mma && dedup_wanted(n_ref, n_cand)).total;
}

int ffr_filter_ex(const void* ref, int64_t n_ref, const void* cand, int64_t n_cand, int32_t dim, int dtype,
                  const float* ref_norm, const float* cand_norm, int metric, float thr, int64_t ref_index_base,
                  uint8_t* keep, int32_t* best_idx, float* best_val, float band_tol, int32_t* band_count,
                  int64_t* band_rows, int64_t band_cap, int flags, void* workspace, size_t ws_bytes,
                  ffr_stream_t stream) {
    (void)ref_norm; (void)cand_norm;     // cosine on pre-normalised fp16 rows needs no norms
    int rc = check_common(ref, n_ref, cand, n_cand, dim, dtype, metric, keep, best_idx);
    if (rc != FFR_OK) return rc;
    if (ffr_device_count() == 0) { set_error("no CUDA device"); return FFR_ERR_CUDA; }
    return filter_core(ref, nullptr, nullptr, nullptr, n_ref, cand, n_cand, dim, dtype, metric, thr, ref_index_base, keep, best_idx,
                       best_val, band_tol, band_count, band_rows, band_cap, flags, workspace, ws_bytes,
                       static_cast<cudaStream_t>(stream));
}

int ffr_filter(const void* ref, int64_t n_ref, const void* cand, int64_t n_cand, int32_t dim, int dtype,
               const float* ref_norm, const float* cand_norm, int metric, float thr, int64_t ref_index_base,
               uint8_t* keep, int32_t* best_idx, float* best_val, void* workspace, size_t ws_bytes,
               ffr_stream_t stream) {
    return ffr_filter_ex(ref, n_ref, cand, n_cand, dim, dtype, ref_norm, cand_norm, metric, thr, ref_index_base, keep,
                         best_idx, best_val, 0.f, nullptr, nullptr, 0, 0, workspace, ws_bytes, stream);
}

size_t ffr_filter_self_workspace_bytes(int64_t n, int64_t n_rows, int32_t dim, int metric) {
    if (n <= 0 || n_rows < 0 || dim <= 0) return 0;
    return self_ws_layout(n, n_rows, dim, metric, dim <= 512 && n > 8).total;     // sized for the tcgen05 path whenever it could run
}

int ffr_filter_self(const float* x, int64_t n, int64_t row_begin, int64_t n_rows, int32_t dim, int metric, int mode,
                    float thr, uint8_t* keep, int32_t* best_idx, float* best_val,
                    float band_tol, int32_t* band_count, int64_t* band_rows, int64_t band_cap,
                    int flags, void* workspace, size_t ws_bytes, ffr_stream_t stream) {
    if (n <= 0) { set_error("n must be > 0 (got %lld)", (long long)n); return FFR_ERR_INVALID; }
    if (dim <= 0) { set_error("dim must be > 0 (got %d)", dim); return FFR_ERR_INVALID; }
    if (row_begin < 0 || n_rows < 0 || row_begin > n - n_rows) {
        set_error("row range [%lld, %lld) is not inside [0, %lld)", (long long)row_begin, (long long)(row_begin + n_rows), (long long)n);
        return FFR_ERR_INVALID;
    }
    if (x == nullptr || (n_rows > 0 && (keep == nullptr || best_idx == nullptr))) { set_error("null pointer argument"); return FFR_ERR_INVALID; }
    if (metric != FFR_METRIC_COSINE && metric != FFR_METRIC_EUCLID) { set_error("unknown metric %d", metric); return FFR_ERR_INVALID; }
    if (mode != FFR_SELF_OTHERS && mode != FFR_SELF_EARLIER) { set_error("unknown self mode %d", mode); return FFR_ERR_INVALID; }
    if (flags & FFR_FLAG_NO_RECHECK) {
        set_error("FFR_FLAG_NO_RECHECK is not supported in self mode (the fp32 re-check decides the masked rows)");
        return FFR_ERR_UNSUPPORTED;
    }
    if (ffr_device_count() == 0) { set_error("no CUDA device"); return FFR_ERR_CUDA; }
    return self_core(x, n, row_begin, n_rows, dim, metric, mode, thr, keep, best_idx, best_val, band_tol, band_count, band_rows,
                     band_cap, flags, workspace, ws_bytes, static_cast<cudaStream_t>(stream));
}

int ffr_filter_stats(const void* workspace, int64_t out[8], ffr_stream_t stream) {
    if (workspace == nullptr || out == nullptr) { set_error("filter_stats: null argument"); return FFR_ERR_INVALID; }
    WsHeader h;
    FFR_CUDA_TRY(cudaMemcpyAsync(&h, workspace, sizeof(h), cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)));
    FFR_CUDA_TRY(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    out[0] = h.recheck_count; out[1] = h.full_count;
    out[2] = g_last.ws == workspace ? g_last.path : -1;
    out[3] = g_last.ws == workspace ? g_last.launches : -1;
    out[4] = h.part_count;
    out[5] = h.refs_scanned;
    out[6] = out[7] = 0;
    return FFR_OK;
}

int ffr_ref_mean_and_thres(const float* ref_feat, int32_t n_ref, int32_t dim, float* mean, float* thres,
                           ffr_stream_t stream) {
    if (ref_feat == nullptr || mean == nullptr || thres == nullptr) { set_error("ref_mean_and_thres: null argument"); return FFR_ERR_INVALID; }
    if (n_ref <= 0 || n_ref > 4096 || dim <= 0 || dim > 8192) { set_error("ref_mean_and_thres: need 0 < n_ref <= 4096, 0 < dim <= 8192"); return FFR_ERR_INVALID; }
    if (ffr_device_count() == 0) { set_error("no CUDA device"); return FFR_ERR_CUDA; }
    return launch_ref_stats(ref_feat, n_ref, dim, mean, thres, static_cast<cudaStream_t>(stream));
}

int ffr_ref_mean_and_thres_batched(const float* ref_feat, const int32_t* offsets, int32_t n_classes, int32_t dim,
                                   float* mean, float* thres, ffr_stream_t stream) {
    if (n_classes < 0 || dim <= 0 || dim > 8192) { set_error("ref_mean_and_thres_batched: need n_classes >= 0, 0 < dim <= 8192"); return FFR_ERR_INVALID; }
    if (n_classes == 0) return FFR_OK;
    if (ref_feat == nullptr || offsets == nullptr || mean == nullptr || thres == nullptr) { set_error("ref_mean_and_thres_batched: null argument"); return FFR_ERR_INVALID; }
    if (ffr_device_count() == 0) { set_error("no CUDA device"); return FFR_ERR_CUDA; }
    return launch_ref_stats_batched(ref_feat, offsets, n_classes, dim, mean, thres, static_cast<cudaStream_t>(stream));
}

int ffr_first_match_stream(float* gallery_feat, float* gallery_bbox, int32_t* gallery_count, int32_t capacity,
                           const float* queries, const float* query_bbox, int32_t n_queries, int32_t dim, int metric,
                           float normal_thres, float harsh_thres, int32_t* match_idx, ffr_stream_t stream) {
    if (capacity <= 0 || n_queries < 0 || dim <= 0 || dim > 8192) { set_error("first_match_stream: need capacity > 0, n_queries >= 0, 0 < dim <= 8192"); return FFR_ERR_INVALID; }
    if (metric != FFR_METRIC_COSINE && metric != FFR_METRIC_EUCLID) { set_error("unknown metric %d", metric); return FFR_ERR_INVALID; }
    if (n_queries == 0) return FFR_OK;
    if (gallery_feat == nullptr || gallery_count == nullptr || queries == nullptr || match_idx == nullptr ||
        (query_bbox != nullptr && gallery_bbox == nullptr)) { set_error("first_match_stream: null argument"); return FFR_ERR_INVALID; }
    if (ffr_device_count() == 0) { set_error("no CUDA device"); return FFR_ERR_CUDA; }
    return launch_first_match_stream(gallery_feat, gallery_bbox, gallery_count, capacity, queries, query_bbox, n_queries, dim,
                                     metric, normal_thres, harsh_thres, match_idx, static_cast<cudaStream_t>(stream));
}

// test hook (not in the public header): tcgen05 kernel on fp16 rows, dumping every score
int ffr_debug_mma_scores(const void* ref16, int64_t n_ref, const void* cand16, int64_t n_cand, int32_t dim_pad,
                         float thr, uint8_t* keep, int32_t* idx, float* val, float* scores, void* workspace,
                         size_t ws_bytes, ffr_stream_t stream) {
    const size_t n = static_cast<size_t>(n_cand);
    const size_t need = 256 + align_up(n * sizeof(RecheckRec), 256) + align_up(n * 4, 256) + align_up(n * 8, 256) +
                        align_up((n / kFullGroup + 1) * 4, 256);
    if (workspace == nullptr || ws_bytes < need) { set_error("debug_mma_scores: workspace needs %zu bytes", need); return FFR_ERR_WORKSPACE; }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    FFR_CUDA_TRY(cudaMemsetAsync(workspace, 0, 256, s));
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    RecheckLists lists;
    lists.hdr = reinterpret_cast<WsHeader*>(ws);
    size_t off = 256;
    lists.recs = reinterpret_cast<RecheckRec*>(ws + off); off += align_up(n * sizeof(RecheckRec), 256);
    lists.full_rows = reinterpret_cast<int32_t*>(ws + off); off += align_up(n * 4, 256);
    lists.full_keys = reinterpret_cast<unsigned long long*>(ws + off); off += align_up(n * 8, 256);
    lists.full_ctr = reinterpret_cast<int32_t*>(ws + off);
    lists.rec_cap = lists.full_cap = n_cand;
    return launch_filter_mma_debug(static_cast<const __half*>(ref16), n_ref, static_cast<const __half*>(cand16), n_cand,
                                   dim_pad, thr, recheck_delta(), keep, idx, val, lists, scores, s);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// host-buffer pipeline
struct ffr_ctx {
    int device;
    int64_t max_ref, chunk;
    int32_t max_dim;
    cudaStream_t s_copy, s_comp;
    cudaEvent_t ev_h2d[2], ev_done[2];
    float* d_ref;
    __half* d_ref16;
    void* d_dedup;             // scratch of the duplicate-reference fold (per call, not per chunk)
    float* d_ebias;            // Euclid: reference bias [pad(max_ref)], its deduplicated copy, squared norms, two scalars
    float* d_ebias_c;
    float* d_ensq;
    float* d_escal;
    float* d_cand[2];
    uint8_t* d_keep[2];
    int32_t* d_idx[2];
    float* d_val[2];
    void* ws[2];
    size_t ws_bytes;
    int64_t launches;
};

extern "C" {

void ffr_ctx_destroy(ffr_ctx* c) {
    if (c == nullptr) return;
    cudaSetDevice(c->device);
    if (c->s_comp) cudaStreamSynchronize(c->s_comp);
    if (c->s_copy) cudaStreamSynchronize(c->s_copy);
    cudaFree(c->d_ref); cudaFree(c->d_ref16); cudaFree(c->d_dedup);
    cudaFree(c->d_ebias); cudaFree(c->d_ebias_c); cudaFree(c->d_ensq); cudaFree(c->d_escal);
    for (int i = 0; i < 2; ++i) {
        cudaFree(c->d_cand[i]); cudaFree(c->d_keep[i]); cudaFree(c->d_idx[i]); cudaFree(c->d_val[i]); cudaFree(c->ws[i]);
        if (c->ev_h2d[i]) cudaEventDestroy(c->ev_h2d[i]);
        if (c->ev_done[i]) cudaEventDestroy(c->ev_done[i]);
    }
    if (c->s_copy) cudaStreamDestroy(c->s_copy);
    if (c->s_comp) cudaStreamDestroy(c->s_comp);
    delete c;
}

int ffr_ctx_create(int device, int64_t max_ref, int64_t chunk_cand, int32_t max_dim, ffr_ctx** out) {
    if (out == nullptr || max_ref <= 0 || chunk_cand <= 0 || max_dim <= 0) { set_error("ctx_create: bad argument"); return FFR_ERR_INVALID; }
    if (ffr_device_count() == 0) { set_error("no CUDA device"); return FFR_ERR_CUDA; }
    ffr_ctx* c = new (std::nothrow) ffr_ctx();
    if (c == nullptr) { set_error("out of host memory"); return FFR_ERR_INVALID; }
    memset(c, 0, sizeof(*c));
    c->device = device; c->max_ref = max_ref; c->chunk = chunk_cand; c->max_dim = max_dim;
#define FFR_CTX_TRY(expr)                                                                          \
    do { cudaError_t _e = (expr); if (_e != cudaSuccess) { int _rc = cuda_fail(_e, #expr); ffr_ctx_destroy(c); return _rc; } } while (0)
    FFR_CTX_TRY(cudaSetDevice(device));
    FFR_CTX_TRY(cudaStreamCreateWithFlags(&c->s_copy, cudaStreamNonBlocking));
    FFR_CTX_TRY(cudaStreamCreateWithFlags(&c->s_comp, cudaStreamNonBlocking));
    const size_t ld = static_cast<size_t>(ffr_padded_dim(max_dim));
    FFR_CTX_TRY(cudaMalloc(&c->d_ref, static_cast<size_t>(max_ref) * max_dim * sizeof(float)));
    FFR_CTX_TRY(cudaMalloc(&c->d_ref16, static_cast<size_t>(max_ref) * ld * 2));
    FFR_CTX_TRY(cudaMalloc(&c->d_dedup, dedup_workspace_bytes(max_ref, static_cast<int32_t>(ld))));
    FFR_CTX_TRY(cudaMalloc(&c->d_ebias, static_cast<size_t>(euclid_bias_len(max_ref)) * sizeof(float)));
    FFR_CTX_TRY(cudaMalloc(&c->d_ebias_c, static_cast<size_t>(euclid_bias_len(max_ref)) * sizeof(float)));
    FFR_CTX_TRY(cudaMalloc(&c->d_ensq, static_cast<size_t>(max_ref) * sizeof(float)));
    FFR_CTX_TRY(cudaMalloc(&c->d_escal, 256));
    // any dim <= max_dim, either metric
    c->ws_bytes = ws_layout(1, chunk_cand, max_dim <= 512 ? max_dim : 512, FFR_DTYPE_F32, true, true, false, true).total;
    if (c->ws_bytes < 4096) c->ws_bytes = 4096;
    for (int i = 0; i < 2; ++i) {
        FFR_CTX_TRY(cudaEventCreateWithFlags(&c->ev_h2d[i], cudaEventDisableTiming));
        FFR_CTX_TRY(cudaEventCreateWithFlags(&c->ev_done[i], cudaEventDisableTiming));
        FFR_CTX_TRY(cudaMalloc(&c->d_cand[i], static_cast<size_t>(chunk_cand) * max_dim * sizeof(float)));
        FFR_CTX_TRY(cudaMalloc(&c->d_keep[i], static_cast<size_t>(chunk_cand)));
        FFR_CTX_TRY(cudaMalloc(&c->d_idx[i], static_cast<size_t>(chunk_cand) * sizeof(int32_t)));
        FFR_CTX_TRY(cudaMalloc(&c->d_val[i], static_cast<size_t>(chunk_cand) * sizeof(float)));
        FFR_CTX_TRY(cudaMalloc(&c->ws[i], c->ws_bytes));
    }
#undef FFR_CTX_TRY
    *out = c;
    return FFR_OK;
}

int ffr_ctx_filter_host(ffr_ctx* c, const float* ref, int64_t n_ref, const float* cand, int64_t n_cand, int32_t dim,
                        int metric, float thr, int64_t ref_index_base, uint8_t* keep, int32_t* best_idx,
                        float* best_val, int flags) {
    if (c == nullptr) { set_error("ctx is null"); return FFR_ERR_INVALID; }
    int rc = check_common(ref, n_ref, cand, n_cand, dim, FFR_DTYPE_F32, metric, keep, best_idx);
    if (rc != FFR_OK) return rc;
    if (n_ref > c->max_ref || dim > c->max_dim) { set_error("ctx sized for n_ref <= %lld, dim <= %d", (long long)c->max_ref, c->max_dim); return FFR_ERR_INVALID; }
    FFR_CUDA_TRY(cudaSetDevice(c->device));
    const int64_t l0 = ffr_launch_count();
    const bool mma = mma_eligible(n_ref, dim, metric, flags);
    FFR_CUDA_TRY(cudaMemcpyAsync(c->d_ref, ref, static_cast<size_t>(n_ref) * dim * sizeof(float), cudaMemcpyHostToDevice, c->s_comp));
    const __half* ref16 = nullptr;
    const int32_t *ref_map = nullptr, *n_unique = nullptr;
    const bool euclid = metric == FFR_METRIC_EUCLID;
    const float* euclid_pre[2] = {c->d_ebias, c->d_escal + 1};
    if (mma) {      // references are normalised / converted (and exact duplicates folded) once, not per chunk
        if (euclid)
            rc = launch_euclid_refs(c->d_ref, n_ref, dim, ffr_padded_dim(dim), c->d_ref16, c->d_ebias, c->d_ensq,
                                    reinterpret_cast<uint32_t*>(c->d_escal), c->d_escal + 1, c->s_comp);
        else
            rc = launch_l2norm(c->d_ref, n_ref, dim, c->d_ref16, ffr_padded_dim(dim), nullptr, nullptr, c->s_comp);
        if (rc != FFR_OK) return rc;
        ref16 = c->d_ref16;
        if (dedup_wanted(n_ref, n_cand)) {
            __half* r16c = nullptr;
            int32_t *map = nullptr, *nuniq = nullptr;
            rc = launch_dedup_refs(c->d_ref, c->d_ref16, n_ref, dim, ffr_padded_dim(dim), c->d_dedup, &r16c, &map, &nuniq, c->s_comp,
                                   euclid ? c->d_ebias : nullptr, c->d_ebias_c);
            if (rc != FFR_OK) return rc;
            ref16 = r16c; ref_map = map; n_unique = nuniq;
            if (euclid) euclid_pre[0] = c->d_ebias_c;
        }
    }
    int64_t i = 0;
    for (int64_t off = 0; off < n_cand; off += c->chunk, ++i) {
        const int b = static_cast<int>(i & 1);
        const int64_t m = (n_cand - off) < c->chunk ? (n_cand - off) : c->chunk;
        if (i >= 2) FFR_CUDA_TRY(cudaStreamWaitEvent(c->s_copy, c->ev_done[b], 0));     // buffer b free again
        FFR_CUDA_TRY(cudaMemcpyAsync(c->d_cand[b], cand + off * dim, static_cast<size_t>(m) * dim * sizeof(float),
                                     cudaMemcpyHostToDevice, c->s_copy));
        FFR_CUDA_TRY(cudaEventRecord(c->ev_h2d[b], c->s_copy));
        FFR_CUDA_TRY(cudaStreamWaitEvent(c->s_comp, c->ev_h2d[b], 0));
        rc = filter_core(c->d_ref, ref16, ref_map, n_unique, n_ref, c->d_cand[b], m, dim, FFR_DTYPE_F32, metric, thr, ref_index_base,
                         c->d_keep[b], c->d_idx[b], c->d_val[b], 0.f, nullptr, nullptr, 0, flags, c->ws[b], c->ws_bytes,
                         c->s_comp, euclid_pre);
        if (rc != FFR_OK) return rc;
        FFR_CUDA_TRY(cudaMemcpyAsync(keep + off, c->d_keep[b], static_cast<size_t>(m), cudaMemcpyDeviceToHost, c->s_comp));
        FFR_CUDA_TRY(cudaMemcpyAsync(best_idx + off, c->d_idx[b], static_cast<size_t>(m) * sizeof(int32_t), cudaMemcpyDeviceToHost, c->s_comp));
        if (best_val != nullptr)
            FFR_CUDA_TRY(cudaMemcpyAsync(best_val + off, c->d_val[b], static_cast<size_t>(m) * sizeof(float), cudaMemcpyDeviceToHost, c->s_comp));
        FFR_CUDA_TRY(cudaEventRecord(c->ev_done[b], c->s_comp));
    }
    FFR_CUDA_TRY(cudaStreamSynchronize(c->s_comp));
    c->launches += ffr_launch_count() - l0;
    return FFR_OK;
}

int64_t ffr_ctx_launch_count(const ffr_ctx* c) { return c ? c->launches : 0; }

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// NCCL gather (dlopen)
namespace {
typedef struct { char internal[128]; } nccl_uid;
typedef void* nccl_comm_t;
typedef int (*pfn_get_uid)(nccl_uid*);
typedef int (*pfn_init_rank)(nccl_comm_t*, int, nccl_uid, int);
typedef int (*pfn_allgather)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t);
typedef int (*pfn_allreduce)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t);
typedef int (*pfn_destroy)(nccl_comm_t);
typedef const char* (*pfn_errstr)(int);
typedef int (*pfn_group)(void);
struct NcclApi {
    void* h = nullptr;
    pfn_get_uid get_uid = nullptr;
    pfn_init_rank init_rank = nullptr;
    pfn_allgather allgather = nullptr;
    pfn_allreduce allreduce = nullptr;
    pfn_destroy destroy = nullptr;
    pfn_errstr errstr = nullptr;
    pfn_group group_start = nullptr, group_end = nullptr;
    bool ok = false;
} g_nccl;
std::mutex g_nccl_mu;

int nccl_load() {
    std::lock_guard<std::mutex> lock(g_nccl_mu);          // (first use from several threads: dlopen + dlsym once)
    if (g_nccl.ok) return FFR_OK;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        g_nccl.h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.h) break;
    }
    if (!g_nccl.h) { set_error("cannot dlopen libnccl.so.2: %s", dlerror()); return FFR_ERR_NCCL; }
    g_nccl.get_uid = reinterpret_cast<pfn_get_uid>(dlsym(g_nccl.h, "ncclGetUniqueId"));
    g_nccl.init_rank = reinterpret_cast<pfn_init_rank>(dlsym(g_nccl.h, "ncclCommInitRank"));
    g_nccl.allgather = reinterpret_cast<pfn_allgather>(dlsym(g_nccl.h, "ncclAllGather"));
    g_nccl.allreduce = reinterpret_cast<pfn_allreduce>(dlsym(g_nccl.h, "ncclAllReduce"));
    g_nccl.destroy = reinterpret_cast<pfn_destroy>(dlsym(g_nccl.h, "ncclCommDestroy"));
    g_nccl.errstr = reinterpret_cast<pfn_errstr>(dlsym(g_nccl.h, "ncclGetErrorString"));
    g_nccl.group_start = reinterpret_cast<pfn_group>(dlsym(g_nccl.h, "ncclGroupStart"));
    g_nccl.group_end = reinterpret_cast<pfn_group>(dlsym(g_nccl.h, "ncclGroupEnd"));
    if (!g_nccl.get_uid || !g_nccl.init_rank || !g_nccl.allgather || !g_nccl.allreduce || !g_nccl.destroy || !g_nccl.group_start || !g_nccl.group_end) {
        set_error("libnccl is missing expected symbols");
        return FFR_ERR_NCCL;
    }
    g_nccl.ok = true;
    return FFR_OK;
}
int nccl_fail(int code, const char* what) {
    set_error("NCCL error %d (%s) at %s", code, g_nccl.errstr ? g_nccl.errstr(code) : "?", what);
    return FFR_ERR_NCCL;
}
}  // namespace

struct ffr_comm {
    nccl_comm_t comm;
    int nranks, rank, device;
};

extern "C" {

int ffr_nccl_unique_id(void* id128) {
    if (id128 == nullptr) { set_error("unique_id: null"); return FFR_ERR_INVALID; }
    int rc = nccl_load();
    if (rc != FFR_OK) return rc;
    nccl_uid uid;
    const int e = g_nccl.get_uid(&uid);
    if (e != 0) return nccl_fail(e, "ncclGetUniqueId");
    memcpy(id128, &uid, sizeof(uid));
    return FFR_OK;
}

int ffr_comm_create(const void* id128, int nranks, int rank, int device, ffr_comm** out) {
    if (id128 == nullptr || out == nullptr || nranks <= 0 || rank < 0 || rank >= nranks) { set_error("comm_create: bad argument"); return FFR_ERR_INVALID; }
    int rc = nccl_load();
    if (rc != FFR_OK) return rc;
    FFR_CUDA_TRY(cudaSetDevice(device));
    nccl_uid uid;
    memcpy(&uid, id128, sizeof(uid));
    ffr_comm* c = new (std::nothrow) ffr_comm();
    if (c == nullptr) { set_error("out of host memory"); return FFR_ERR_INVALID; }
    c->nranks = nranks; c->rank = rank; c->device = device; c->comm = nullptr;
    const int e = g_nccl.init_rank(&c->comm, nranks, uid, rank);
    if (e != 0) { delete c; return nccl_fail(e, "ncclCommInitRank"); }
    *out = c;
    return FFR_OK;
}

void ffr_comm_destroy(ffr_comm* c) {
    if (c == nullptr) return;
    if (c->comm && g_nccl.ok) g_nccl.destroy(c->comm);
    delete c;
}

size_t ffr_allgather_workspace_bytes(int nranks, int64_t m_local) {
    if (nranks <= 0 || m_local < 0) return 0;
    const size_t m_pad = (static_cast<size_t>(m_local) + 15) / 16 * 16;
    return (static_cast<size_t>(nranks) + 1) * m_pad * 5 + 256;
}

int ffr_allgather_results(ffr_comm* c, const uint8_t* keep_local, const int32_t* idx_local, int64_t m_local,
                          uint8_t* keep_all, int32_t* idx_all, void* workspace, size_t ws_bytes, ffr_stream_t stream) {
    if (c == nullptr || keep_local == nullptr || idx_local == nullptr || keep_all == nullptr || idx_all == nullptr) { set_error("allgather: null argument"); return FFR_ERR_INVALID; }
    if (m_local < 0) { set_error("allgather: m_local < 0"); return FFR_ERR_INVALID; }
    if (m_local == 0) return FFR_OK;
    const size_t need = ffr_allgather_workspace_bytes(c->nranks, m_local);
    if (workspace == nullptr || ws_bytes < need) { set_error("allgather: workspace needs %zu bytes", need); return FFR_ERR_WORKSPACE; }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t m_pad = (m_local + 15) / 16 * 16;
    uint8_t* send = static_cast<uint8_t*>(workspace);
    uint8_t* recv = send + static_cast<size_t>(m_pad) * 5;
    int rc = launch_pack_results(keep_local, idx_local, m_local, m_pad, send, s);
    if (rc != FFR_OK) return rc;
    const int e = g_nccl.allgather(send, recv, static_cast<size_t>(m_pad) * 5, /*ncclUint8*/ 1, c->comm, s);
    if (e != 0) return nccl_fail(e, "ncclAllGather");
    return launch_unpack_results(recv, m_local, m_pad, c->nranks, keep_all, idx_all, s);
}

int ffr_allgather_results_inplace(ffr_comm* c, uint8_t* keep_all, int32_t* idx_all, int64_t m_local, ffr_stream_t stream) {
    if (c == nullptr || keep_all == nullptr || idx_all == nullptr) { set_error("allgather_inplace: null argument"); return FFR_ERR_INVALID; }
    if (m_local < 0) { set_error("allgather_inplace: m_local < 0"); return FFR_ERR_INVALID; }
    if (m_local == 0) return FFR_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t m = static_cast<size_t>(m_local);
    // the two in-place gathers are fused by the group into ONE NCCL launch; this library launches no kernel of its own
    int e = g_nccl.group_start();
    if (e != 0) return nccl_fail(e, "ncclGroupStart");
    e = g_nccl.allgather(idx_all + static_cast<size_t>(c->rank) * m, idx_all, m, /*ncclInt32*/ 2, c->comm, s);
    if (e == 0) e = g_nccl.allgather(keep_all + static_cast<size_t>(c->rank) * m, keep_all, m, /*ncclUint8*/ 1, c->comm, s);
    const int e2 = g_nccl.group_end();
    if (e != 0) return nccl_fail(e, "ncclAllGather (in place)");
    if (e2 != 0) return nccl_fail(e2, "ncclGroupEnd");
    return FFR_OK;
}

size_t ffr_allreduce_best_workspace_bytes(int64_t n_cand) {
    if (n_cand < 0) return 0;
    const size_t b = align_up(static_cast<size_t>(n_cand) * sizeof(unsigned long long), 256);
    return b > 0 ? b : 256;
}

int ffr_allreduce_best(ffr_comm* c, const float* ref_local, int64_t n_ref_local, int64_t ref_index_base, const float* cand,
                       int64_t n_cand, int32_t dim, int metric, float thr, uint8_t* keep, int32_t* best_idx, float* best_val,
                       float band_tol, int32_t* band_count, int64_t* band_rows, int64_t band_cap, void* workspace,
                       size_t ws_bytes, ffr_stream_t stream) {
    if (c == nullptr) { set_error("allreduce_best: comm is null"); return FFR_ERR_INVALID; }
    if (n_ref_local < 0 || n_cand < 0 || dim <= 0) {
        set_error("allreduce_best: need n_ref_local >= 0, n_cand >= 0, dim > 0 (got %lld, %lld, %d)", (long long)n_ref_local,
                  (long long)n_cand, dim);
        return FFR_ERR_INVALID;
    }
    if (ref_index_base < 0 || ref_index_base + n_ref_local > static_cast<int64_t>(INT32_MAX)) {
        set_error("allreduce_best: global reference indices [%lld, %lld) do not fit int32", (long long)ref_index_base,
                  (long long)(ref_index_base + n_ref_local));
        return FFR_ERR_INVALID;
    }
    if (metric != FFR_METRIC_COSINE && metric != FFR_METRIC_EUCLID) { set_error("unknown metric %d", metric); return FFR_ERR_INVALID; }
    if ((n_ref_local > 0 && ref_local == nullptr) ||
        (n_cand > 0 && (cand == nullptr || keep == nullptr || best_idx == nullptr))) {
        set_error("allreduce_best: null pointer argument");
        return FFR_ERR_INVALID;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (band_count != nullptr) FFR_CUDA_TRY(cudaMemsetAsync(band_count, 0, sizeof(int32_t), s));
    if (n_cand == 0) return FFR_OK;
    const size_t need = ffr_allreduce_best_workspace_bytes(n_cand);
    if (workspace == nullptr || ws_bytes < need) {
        set_error("allreduce_best: workspace needs %zu bytes, got %zu", need, workspace ? ws_bytes : (size_t)0);
        return FFR_ERR_WORKSPACE;
    }
    if (reinterpret_cast<uintptr_t>(workspace) & 7) { set_error("allreduce_best: workspace must be 8-byte aligned"); return FFR_ERR_INVALID; }
    unsigned long long* keys = static_cast<unsigned long long*>(workspace);
    int rc = launch_best_keys(ref_local, n_ref_local, ref_index_base, cand, n_cand, dim, metric, best_idx, keys, s);
    if (rc != FFR_OK) return rc;
    const int e = g_nccl.allreduce(keys, keys, static_cast<size_t>(n_cand), /*ncclUint64*/ 5, /*ncclMax*/ 2, c->comm, s);
    if (e != 0) return nccl_fail(e, "ncclAllReduce");
    return launch_emit_keys(keys, n_cand, metric, thr, keep, best_idx, best_val, band_tol, band_count, band_rows, band_cap, s);
}

}  // extern "C"

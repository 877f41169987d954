/*
 * ffr.h -- C ABI of the B200-native similar-face-filtering hot path ("ffr" = face filter by reference).
 *
 * The reference (SamSamhuns/face_detection_and_recognition) is pure Python and has NO FFI / plugin
 * interface for this path: the arithmetic is inline NumPy in
 *     similar_face_filtering/filter_faces_using_reference.py:85-99   (mean vector + max-dist threshold)
 *     similar_face_filtering/filter_faces_using_reference.py:186-189 (per-row Euclid keep test)
 *     face_detection_and_extraction/face_extraction/extract_and_label_faces_from_dataset.py:101-116
 *                                                                    (per-pair cosine/Euclid + threshold scan)
 *     face_detection_and_extraction/modules/mobile_facenet/mobile_facenet.py:30-33  (l2_norm)
 *     face_detection_and_extraction/face_extraction/extract_and_clean_imdb_wiki_faces.py:146 (NumPy L2-normalise)
 * so the entry points below are what a ctypes binding added to those call sites would bind
 * (INTEGRATION.md shows the stub).  Every entry point cites the reference expression it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / CUDA types in the signatures (ffr_stream_t is a
 *     cudaStream_t passed as void*; NULL = the legacy default stream).
 *   - "device" pointers are caller-owned CUDA device memory, row-major, contiguous, 16-byte aligned.
 *   - every device-pointer call is asynchronous on the given stream and allocates nothing: scratch
 *     memory is an explicit workspace sized by the matching *_workspace_bytes query.
 *   - return 0 on success, a negative FFR_ERR_* code otherwise; ffr_last_error() gives the
 *     thread-local message.  There is no CPU fallback: without a CUDA device every compute entry
 *     point fails with FFR_ERR_CUDA.
 */
#ifndef FFR_H_
#define FFR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FFR_ABI_VERSION 1

#define FFR_OK               0
#define FFR_ERR_INVALID     -1   /* bad argument (null pointer, non-positive size, misalignment) */
#define FFR_ERR_CUDA        -2   /* CUDA runtime / driver error, or no device */
#define FFR_ERR_WORKSPACE   -3   /* workspace missing or too small */
#define FFR_ERR_UNSUPPORTED -4   /* shape / dtype / metric combination not implemented */
#define FFR_ERR_NCCL        -5   /* NCCL could not be loaded or returned an error */

#define FFR_METRIC_COSINE 0      /* best = max_i (r_i.c)/(|r_i||c|), keep = best >= thr  (extract_and_label...:106) */
#define FFR_METRIC_EUCLID 1      /* best = min_i |c - r_i|,          keep = best <= thr  (filter_faces...:189, extract_and_label...:104) */

#define FFR_DTYPE_F32 0          /* raw fp32 embeddings; the op normalises internally */
#define FFR_DTYPE_F16 1          /* rows already L2-normalised + converted by ffr_l2norm_rows_f32 (leading dim = ffr_padded_dim).
                                    There are no fp32 rows to re-check against: keep / best_idx are then exact in fp16-OPERAND space
                                    (the index carries the row's largest fp16-operand score, ties -> first), i.e. they can differ from
                                    the fp32 decision for pairs closer than ~1.5e-4; best_val is within 1e-3 as always */

/* flags for ffr_filter_ex */
#define FFR_FLAG_FORCE_FP32   1  /* use the exact fp32 CUDA-core kernel whatever the shape */
#define FFR_FLAG_FORCE_MMA    2  /* use the tcgen05 kernel (dim <= 512) whatever n_ref (euclid: n_ref > 8 still required) */
#define FFR_FLAG_NO_RECHECK   4  /* skip the fp32 re-check of near-tie / near-threshold rows (benchmarking only): decisions as for FFR_DTYPE_F16 */

typedef void* ffr_stream_t;      /* cudaStream_t */
typedef struct ffr_ctx  ffr_ctx; /* host-buffer pipeline context (streams, staging, workspace) */
typedef struct ffr_comm ffr_comm;/* one NCCL communicator + scratch */

int         ffr_abi_version(void);
const char* ffr_last_error(void);
const char* ffr_build_info(void);            /* "sm_100a; nvcc x.y; ..." */
int         ffr_device_count(void);           /* 0 when no CUDA device is visible */

/* leading dimension (in elements) of the fp16 rows the tensor-core kernel consumes: dim rounded up to 64 */
int32_t ffr_padded_dim(int32_t dim);

/* ---- K1: row L2-normalisation ---------------------------------------------------------------
 * y[i,:] = x[i,:] / |x[i,:]|_2   (no epsilon)      replaces  mobile_facenet.py:30-33  l2_norm
 *                                                            extract_and_clean_imdb_wiki_faces.py:146
 * and supplies the denominators of extract_and_label_faces_from_dataset.py:106.
 * Any of the three outputs may be NULL.  y_f16 has leading dimension y_f16_ld >= dim (columns
 * dim..y_f16_ld-1 are written as zeros); y_f32 and x may alias.  norms[i] = |x[i,:]|_2. */
int ffr_l2norm_rows_f32(const float* x, int64_t rows, int32_t dim,
                        void* y_f16, int32_t y_f16_ld, float* y_f32, float* norms,
                        ffr_stream_t stream);

/* ---- K2/K2s/K3: fused reference x candidate filter -------------------------------------------
 * For every candidate row c of cand[n_cand, dim]:
 *   cosine:  best = max_i (r_i.c)/(|r_i||c|)   idx = first argmax   keep = best >= thr
 *   euclid:  best = min_i |c - r_i|_2          idx = first argmin   keep = best <= thr
 * replaces the per-row test  filter_faces_using_reference.py:186-189 (euclid, n_ref = 1, ref = mean
 * vector) and the per-pair scan extract_and_label_faces_from_dataset.py:101-116; the n_ref x n_cand
 * similarity matrix is never materialised.
 *   ref, cand      device, dtype FFR_DTYPE_F32 (dim floats per row) or FFR_DTYPE_F16 (see above)
 *   ref_norm,cand_norm  device, only read with FFR_DTYPE_F16 (may be NULL for cosine)
 *   ref_index_base added to every best_idx (global index of ref row 0)
 *   keep u8[n_cand], best_idx i32[n_cand], best_val f32[n_cand]   device outputs (best_val may be NULL)
 * ffr_filter_ex additionally lists the tolerance band: rows with |best - thr| <= band_tol are appended
 * (unordered) to band_rows[0..band_cap) and counted in *band_count (device int32; count may exceed cap); `best` is the
 * fp32 re-checked score, or the fp16-operand score where no re-check runs (FFR_DTYPE_F16, FFR_FLAG_NO_RECHECK).
 * Bit-identical reference rows are folded internally (a later copy can never be the first arg-best); best_idx always
 * refers to the caller's row numbering.
 * Euclid on the tensor cores: with n_ref > 8, dim <= 512, FFR_DTYPE_F32, the re-check on (no FFR_FLAG_NO_RECHECK, no
 * FFR_FLAG_FORCE_FP32) and a GPU whose SMs pair up (cta_group::2), euclid runs K1 + K2 (fp16 dot products plus a per-reference
 * bias) + K3 (fp32 distances of the near ties) + a value pass; otherwise the exact fp32 kernel K2s.  Contract: best_idx equals
 * the FFR_FLAG_FORCE_FP32 result except on rows whose two smallest distances differ by < 1e-6 relative (fp32 ties); keep and
 * best_val are bit-identical to it wherever best_idx agrees; the band list is exact.  FFR_DTYPE_F16 rows are refused for
 * euclid (FFR_ERR_UNSUPPORTED). */
size_t ffr_filter_workspace_bytes(int64_t n_ref, int64_t n_cand, int32_t dim, int dtype, int metric);

int ffr_filter(const void* ref, int64_t n_ref, const void* cand, int64_t n_cand, int32_t dim, int dtype,
               const float* ref_norm, const float* cand_norm, int metric, float thr, int64_t ref_index_base,
               uint8_t* keep, int32_t* best_idx, float* best_val,
               void* workspace, size_t ws_bytes, ffr_stream_t stream);

int ffr_filter_ex(const void* ref, int64_t n_ref, const void* cand, int64_t n_cand, int32_t dim, int dtype,
                  const float* ref_norm, const float* cand_norm, int metric, float thr, int64_t ref_index_base,
                  uint8_t* keep, int32_t* best_idx, float* best_val,
                  float band_tol, int32_t* band_count, int64_t* band_rows, int64_t band_cap,
                  int flags, void* workspace, size_t ws_bytes, ffr_stream_t stream);

/* ---- self mode: each row's best match among the OTHER rows of the same set ------------------------------------
 * Near-duplicate search inside one embedding set (the IMDB-WIKI cleaner's question; the tracker's check_if_face_exists asked
 * one query at a time).  x[n, dim] fp32 (device) is both the candidate and the reference matrix: the candidates are rows
 * [row_begin, row_begin + n_rows) (so candidate-axis sharding works unchanged), the references all n rows, and best_idx is a
 * global row index of x.  keep / best_idx / best_val / the band hold n_rows entries, local to the row range.
 *   FFR_SELF_OTHERS   best over every reference i != j (leave-one-out)
 *   FFR_SELF_EARLIER  best over i < j: with keep = 1 row j is a near-duplicate of an EARLIER row, so dropping exactly the kept
 *                     rows leaves the first occurrence of every group
 * A row with no eligible reference (row 0 in EARLIER, or n = 1): keep = 0, best_idx = -1, best_val = -inf (cosine) / +inf
 * (Euclid), never in the band.  Bit-identical rows are NOT folded: they are what the caller is looking for.
 * Metric, threshold, first-occurrence ties, band and precision contract are ffr_filter_ex's applied to the masked problem
 * (the Euclid rule included: best_idx equals the FFR_FLAG_FORCE_FP32 result except on fp32 ties, keep / best_val bit-identical
 * to it wherever best_idx agrees).  Tensor cores when n > 8, dim <= 512, the re-check is on and the GPU runs cta_group::2;
 * otherwise (and with FFR_FLAG_FORCE_FP32) the exact fp32 kernel K2s in its self form.  FFR_FLAG_NO_RECHECK is refused
 * (FFR_ERR_UNSUPPORTED), a row range outside [0, n) too (FFR_ERR_INVALID).  ffr_filter_stats works on this workspace. */
#define FFR_SELF_OTHERS  0
#define FFR_SELF_EARLIER 1
size_t ffr_filter_self_workspace_bytes(int64_t n, int64_t n_rows, int32_t dim, int metric);
int ffr_filter_self(const float* x, int64_t n, int64_t row_begin, int64_t n_rows, int32_t dim, int metric, int mode,
                    float thr, uint8_t* keep, int32_t* best_idx, float* best_val,
                    float band_tol, int32_t* band_count, int64_t* band_rows, int64_t band_cap,
                    int flags, void* workspace, size_t ws_bytes, ffr_stream_t stream);

/* statistics of the last ffr_filter* call that used this workspace (device->host copy, synchronises
 * the stream): out[0] = rows re-checked in fp32 against their two or three leading references (near-tie or
 * near-threshold), out[1] = rows that needed the full fp32 rescan, out[2] = path taken (0 fp32 CUDA-core,
 * 1 tcgen05), out[3] = kernels launched, out[4] = rows re-checked against one 128-reference part, out[5] = reference
 * rows the tensor-core kernel scanned (< n_ref when bit-identical reference rows were folded), out[6..7] = 0. */
int ffr_filter_stats(const void* workspace, int64_t out[8], ffr_stream_t stream);

/* ---- K5: reference statistics -----------------------------------------------------------------
 * mean[d] = mean_i ref_feat[i,d];  *thres = max_i |mean - ref_feat[i,:]|_2
 * replaces filter_faces_using_reference.py:85-99.  n_ref <= 4096.  mean f32[dim], thres f32[1]: device. */
int ffr_ref_mean_and_thres(const float* ref_feat, int32_t n_ref, int32_t dim,
                           float* mean, float* thres, ffr_stream_t stream);

/* all classes in one launch: class c owns rows offsets[c] .. offsets[c+1]-1 of ref_feat (offsets: device int32
 * [n_classes + 1]); mean f32[n_classes, dim], thres f32[n_classes].  Same arithmetic per class as above. */
int ffr_ref_mean_and_thres_batched(const float* ref_feat, const int32_t* offsets, int32_t n_classes, int32_t dim,
                                   float* mean, float* thres, ffr_stream_t stream);

/* ---- streaming first-match gallery scan ("next" row: the reference's face tracker) -------------------
 * replaces Net.check_if_face_exists + add_face, face_extraction/extract_and_label_faces_from_dataset.py:101-121.
 * Queries are processed IN ORDER against a device-resident gallery (feat f32[capacity, dim], bbox f32[capacity, 4],
 * *gallery_count entries in use): the first entry i (ascending) with
 *     (dist < normal_thres and iou(bbox_i, query_bbox) > 0.1) or dist < harsh_thres
 * is overwritten by the query and match_idx[q] = i; otherwise the query is appended at position p = old count and
 * match_idx[q] = -1 - p (INT32_MIN if the gallery is full).  dist = 1 - cos (FFR_METRIC_COSINE, :106) or the Euclid
 * distance (FFR_METRIC_EUCLID, :104).  query_bbox may be NULL (iou = 0: only the harsh threshold can match). */
int ffr_first_match_stream(float* gallery_feat, float* gallery_bbox, int32_t* gallery_count, int32_t capacity,
                           const float* queries, const float* query_bbox, int32_t n_queries, int32_t dim, int metric,
                           float normal_thres, float harsh_thres, int32_t* match_idx, ffr_stream_t stream);

/* ---- host-buffer ("plugin") entry points -----------------------------------------------------
 * Same semantics as ffr_filter with HOST pointers: candidates are streamed host->device in chunks on
 * one stream while the previous chunk is filtered on another; results are copied back.  Pinned host
 * buffers overlap fully; pageable ones work but serialise.  Synchronous (returns when results are in
 * the host arrays). */
int  ffr_ctx_create(int device, int64_t max_ref, int64_t chunk_cand, int32_t max_dim, ffr_ctx** out);
void ffr_ctx_destroy(ffr_ctx* ctx);
int  ffr_ctx_filter_host(ffr_ctx* ctx, const float* ref, int64_t n_ref, const float* cand, int64_t n_cand,
                         int32_t dim, int metric, float thr, int64_t ref_index_base,
                         uint8_t* keep, int32_t* best_idx, float* best_val, int flags);
/* number of this library's kernel launches issued through ctx so far (for bench accounting) */
int64_t ffr_ctx_launch_count(const ffr_ctx* ctx);
/* process-wide count of this library's kernel launches */
int64_t ffr_launch_count(void);

/* ---- K4: multi-GPU gather of the per-candidate result (one rank per GPU) -----------------------
 * Candidates are sharded contiguously, m_local rows per rank (equal on every rank; pad the last).
 * keep_all / idx_all receive nranks * m_local entries in rank order.  One ncclAllGather of the
 * packed {idx i32, keep u8} records over NVLink; NCCL is dlopen'ed (libnccl.so.2) on first use. */
int  ffr_nccl_unique_id(void* id128);                        /* 128 bytes, call on rank 0 and broadcast */
int  ffr_comm_create(const void* id128, int nranks, int rank, int device, ffr_comm** out);
void ffr_comm_destroy(ffr_comm* comm);
size_t ffr_allgather_workspace_bytes(int nranks, int64_t m_local);
int  ffr_allgather_results(ffr_comm* comm, const uint8_t* keep_local, const int32_t* idx_local, int64_t m_local,
                           uint8_t* keep_all, int32_t* idx_all, void* workspace, size_t ws_bytes,
                           ffr_stream_t stream);
/* In-place form (no pack / unpack kernels, no workspace): this rank's ffr_filter already wrote its m_local results at
 * keep_all + rank * m_local and idx_all + rank * m_local (pass those as the filter's keep / best_idx outputs); the two
 * in-place ncclAllGather calls are grouped into ONE NCCL launch that fills in everybody else's slices. */
int  ffr_allgather_results_inplace(ffr_comm* comm, uint8_t* keep_all, int32_t* idx_all, int64_t m_local,
                                   ffr_stream_t stream);

/* ---- gallery sharded over ranks: merge of the per-rank best matches ---------------------------------------------
 * The references (the gallery) are split across ranks, the candidates (probes) replicated.  Each rank has run ffr_filter* on
 * its shard ref_local[n_ref_local, dim] with ref_index_base = the global index of its row 0, and passes that result's best_idx
 * (device i32[n_cand], global indices) in; on return every rank holds the identical result for the WHOLE gallery in keep,
 * best_idx and best_val (best_val may be NULL), plus the band (|best - thr| <= band_tol, as ffr_filter_ex).
 *   1. one kernel recomputes the fp32 value of the rank's winner from ref_local and cand (cosine: K3's arithmetic; Euclid: the
 *      distance K2s computes) -- the filter's best_val may be an fp16-operand score, which cannot be compared across ranks --
 *      and packs the key (orderable(v) << 32) | ~idx, v = score (cosine) or -distance (Euclid);
 *   2. one in-place ncclAllReduce(ncclUint64, ncclMax) over n_cand keys: best value, then the smallest global index (the first
 *      occurrence over the whole gallery);
 *   3. one kernel writes best_idx / best_val, decides keep from thr and appends the band.
 * A rank with an empty shard (n_ref_local = 0, ref_local may be NULL; it runs no filter) contributes the identity key 0, as does
 * a row whose best_idx lies outside [ref_index_base, ref_index_base + n_ref_local).  A row no rank has a reference for gets
 * keep 0, best_idx -1, best_val -inf (cosine) / +inf (Euclid).  Precision: the one-GPU gallery contract over the whole gallery
 * (best_idx equal except on fp32 ties, keep exact outside |best - thr| < 1e-6, Euclid keep / best_val bit-identical to the
 * one-GPU call wherever best_idx agrees); best_val is always the fp32 value of the returned reference.  Every rank must call
 * with the same n_cand, metric, thr and band arguments.  The workspace holds n_cand 64-bit keys. */
size_t ffr_allreduce_best_workspace_bytes(int64_t n_cand);
int  ffr_allreduce_best(ffr_comm* comm, const float* ref_local, int64_t n_ref_local, int64_t ref_index_base, const float* cand,
                        int64_t n_cand, int32_t dim, int metric, float thr, uint8_t* keep, int32_t* best_idx, float* best_val,
                        float band_tol, int32_t* band_count, int64_t* band_rows, int64_t band_cap,
                        void* workspace, size_t ws_bytes, ffr_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* FFR_H_ */

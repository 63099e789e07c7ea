/*
 * hm_matcher.h - C ABI of the B200-native Hamming brute-force matcher.
 *
 * Drop-in boundary for ONE path of ViV99/slam-experiments: the brute-force
 * Hamming k-nearest-neighbour matching of 256-bit ORB descriptors that
 * /root/reference/feature_matchers.py:32-44 performs through
 * cv2.BFMatcher(NORM_HAMMING).  The reference has no FFI of its own (it calls
 * the opencv-python wheel), so the entry points below are what a binding for
 * this path would bind; INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *  - plain C: pointers, sizes, no C++ types, no exceptions across the boundary;
 *  - every function returns an hm_status (0 = ok, <0 = error);
 *    hm_last_error() returns a thread-local description of the last failure;
 *  - all data pointers are DEVICE pointers unless the name ends in _host;
 *    the library never allocates or frees caller-visible memory: inputs,
 *    outputs and workspace are caller-allocated (torch tensors in the Python
 *    host) and nothing is retained after return;
 *  - functions enqueue on `stream` (a cudaStream_t passed as void*, NULL =
 *    legacy default stream) and return without synchronising;
 *  - descriptors are rows of HM_DESC_BYTES = 32 bytes (256 bits); row strides
 *    are in BYTES, must be multiples of 16, and base pointers 16-byte aligned;
 *  - "query" / "train" follow cv2: bf.match(query, train).  The reference
 *    passes its `source_descriptors` as train (feature_matchers.py:39).
 *
 * Result format: packed 64-bit keys
 *      key = (uint64)distance << 32 | trainIdx          (distance in 0..256)
 *  so that unsigned min() over keys is cv2's order: ascending distance, ties
 *  to the lowest trainIdx (BFMatcher::knnMatchImpl, matchers.cpp; SURVEY.md
 *  E2).  A missing neighbour (Nt < 2) is HM_NO_MATCH.
 */
#ifndef HM_MATCHER_H_
#define HM_MATCHER_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define HM_API __declspec(dllexport)
#else
#define HM_API __attribute__((visibility("default")))
#endif

#define HM_ABI_VERSION 4
#define HM_DESC_BYTES 32
#define HM_DESC_BITS 256
#define HM_NO_MATCH 0xFFFFFFFFFFFFFFFFull
/* one descriptor expanded to +/-1 int8 (HM_VARIANT_I8) / +/-1 e2m1 4-bit floats (HM_VARIANT_F4) */
#define HM_PREPARED_ROW_BYTES 256
#define HM_PREPARED_F4_ROW_BYTES 128
/* the tensor-core core HM_VARIANT_AUTO resolves to (ncu evidence in DESIGN.md) */
#define HM_DEFAULT_TENSOR_VARIANT 3
/* prepared images are padded to whole tiles of this many rows */
#define HM_PREPARED_TILE_ROWS 256
/* Measurement aid: the tensor-core k-NN kernels leave four int64 at this byte offset of the workspace they were given --
 * %globaltimer (ns) and clock64 (SM cycles) of their first CTA at entry and at exit.  (cycles / ns) is the SM clock the
 * kernel really ran at; bench.py reports it next to NVML's figure.  Not part of the data path. */
#define HM_WS_CLOCK_PROBE_OFFSET 64

typedef enum hm_status {
    HM_OK = 0,
    HM_ERR_INVALID_ARGUMENT = -1, /* cv2 raises cv2.error(-215) for these (batch_distance.cpp:274,282) */
    HM_ERR_CUDA = -2,             /* a CUDA runtime call failed; see hm_last_error() */
    HM_ERR_WORKSPACE = -3,        /* workspace pointer NULL or smaller than its sizing function reports
                                     (hm_db_mutual_flags: also when not 256-byte aligned) */
    HM_ERR_UNSUPPORTED = -4,      /* shape / variant outside the supported domain */
    HM_ERR_NO_DEVICE = -5         /* no sm_100 device visible: there is NO CPU fallback */
} hm_status;

typedef enum hm_variant {
    HM_VARIANT_AUTO = 0, /* static per-shape table baked from ncu evidence (DESIGN.md) */
    HM_VARIANT_POPC = 1, /* (a) LOP3 XOR + POPC on 32-bit words */
    HM_VARIANT_I8 = 2,   /* (b) tcgen05 kind::i8 GEMM on +/-1 expansion, H = (256 - dot) / 2 */
    HM_VARIANT_F4 = 3    /* (b') same GEMM through tcgen05 kind::mxf4: +/-1 as e2m1, unit block scales, exact
                            fp32 dot products, twice the kind::i8 issue rate and half the operand bytes */
} hm_variant;

/* flags of hm_filter_matches / hm_match_fused */
#define HM_FLAG_RATIO 1u          /* Lowe ratio test: keep iff d1 < ratio_lut[d2] (needs 2 neighbours) */
#define HM_FLAG_MUTUAL 2u         /* cross-check: keep iff q is t's best query too (cv2 crossCheck=True) */
#define HM_FLAG_DIST_THRESHOLD 4u /* reference filter: d < max(2*min_d, thr), feature_matchers.py:41-43 */
/* Combination rule: the three tests are independent predicates on a query row's forward neighbours, and a match is
 * kept iff every requested one holds.  min_d of the distance filter is taken over ALL forward best matches (what
 * feature_matchers.py:41 sees: the reference's matcher has crossCheck=False and no ratio test), not over the
 * survivors of RATIO / MUTUAL; the reference itself never combines them (tested: test_fused_pipeline_and_batched_vs_oracle, case ratio 0.9 + mutual + thr 64.5). */

/* ---- introspection ------------------------------------------------------------------ */
HM_API int hm_version(void);
HM_API const char* hm_last_error(void);
/* number of SMs of the current device, or an hm_status (<0) */
HM_API int hm_device_sm_count(void);
/* the variant HM_VARIANT_AUTO resolves to for this shape */
HM_API int hm_select_variant(int64_t nq, int64_t nt, int batch);
/* which kernel (and grid) hm_knn2* launches for this shape, as text: "hm_f4_knn2_floor_kernel grid=(8,37,1)
 * cluster=2 tiles_per_cta=1730"; for bench lines and profiles, not part of the data path */
HM_API int hm_describe_launch(int64_t nq, int64_t nt, int batch, int variant, char* buf, size_t buf_bytes);
/* scratch bytes hm_knn2* / hm_match_fused* need for this shape (variant may be AUTO) */
HM_API size_t hm_workspace_bytes(int64_t nq, int64_t nt, int batch, int variant);

/* ---- measurement hook ---------------------------------------------------------------- */
/* When both are non-NULL (cudaEvent_t as void*), the NEXT dominant-kernel launch of this thread
 * (hm_popc_knn2_kernel, hm_i8_knn2*_kernel or hm_f4_knn2*_kernel: the forward k-NN of a pipeline call) records
 * `start` immediately before and `stop` immediately after it on the call's stream, so bench.py can time that
 * kernel alone with CUDA events; call again to re-arm.  Pass NULLs to switch it off.  Not part of the data path. */
HM_API void hm_profile_events(void* start_event, void* stop_event);

/* ---- k-NN core: replaces cv2.BFMatcher.knnMatch(query, train, k=2) and, through key[0],
 *      cv2.BFMatcher.match(query, train) = /root/reference/feature_matchers.py:39 -------- */
/* out_keys[nq][2]; train_base is added to every trainIdx (global row id of a shard's first row) */
HM_API int hm_knn2(const uint8_t* query, int64_t nq, int64_t q_stride,
                   const uint8_t* train, int64_t nt, int64_t t_stride,
                   uint64_t train_base, uint64_t* out_keys,
                   int variant, void* workspace, size_t workspace_bytes, void* stream);

/* `batch` independent problems of identical shape; problem b reads
 * query + b*q_batch_stride and train + b*t_batch_stride (bytes) and writes
 * out_keys[b][nq][2].  Overlapping windows are allowed (frame i+1 vs frame i of
 * one resident sequence: /root/reference/frontend.py:185-187). */
HM_API int hm_knn2_batched(const uint8_t* query, int64_t nq, int64_t q_stride, int64_t q_batch_stride,
                           const uint8_t* train, int64_t nt, int64_t t_stride, int64_t t_batch_stride,
                           int batch, uint64_t* out_keys,
                           int variant, void* workspace, size_t workspace_bytes, void* stream);

/* Resident database + packed query: the call a keyframe database makes per query batch.  `train_prepared` is an image
 * written by hm_prepare(); `query` are plain descriptors (nq rows, q_stride bytes apart).  With HM_VARIANT_F4 the k-NN
 * kernel expands the query rows itself (one launch per call); with HM_VARIANT_I8 the query is expanded into the tail of
 * the workspace first.  Workspace: hm_resident_workspace_bytes(nq, nt, variant).  Same result as
 * cv2.BFMatcher.knnMatch(query, train, k=2) (/root/reference/feature_matchers.py:39 for key[0]). */
HM_API size_t hm_resident_workspace_bytes(int64_t nq, int64_t nt, int variant);
HM_API int hm_knn2_resident(const uint8_t* query, int64_t nq, int64_t q_stride,
                            const void* train_prepared, int64_t nt, uint64_t train_base, uint64_t* out_keys,
                            int variant, void* workspace, size_t workspace_bytes, void* stream);
/* the same with the cross-GPU exchange of hm_knn2_prepared_exchange folded into the kernel's last-CTA merge */
HM_API int hm_knn2_resident_exchange(const uint8_t* query, int64_t nq, int64_t q_stride,
                                     const void* train_prepared, int64_t nt, uint64_t train_base,
                                     int world, int rank, void* const* peer_buffers_host, int64_t max_rows,
                                     uint32_t epoch, uint64_t* out_keys, int variant, void* workspace,
                                     size_t workspace_bytes, void* stream);

/* ---- keyframe database: search a selection of the train rows ------------------------------------------------------
 * A selection is a list of n_runs RUNS [lo, hi) of train rows (shard-local), ascending, disjoint and non-empty, with
 * hi <= nt < 2^32.  The result equals hm_knn2 over the concatenation of the selected rows, with every trainIdx mapped
 * back to its row (+ train_base): the stable top-2 over the selected rows, ties to the lowest row.  Unselected rows
 * cost nothing beyond the 128-row tiles a run starts or ends in.
 *  runs_host[n_runs][2]  host array (lo, hi): validated (HM_ERR_INVALID_ARGUMENT before any launch for unsorted,
 *                        overlapping, empty or out-of-range runs) and planned from
 *  runs_dev[n_runs][4]   device array the caller uploads with the same runs: lo, hi, the 128-row tiles the runs before
 *                        it touch (sum of ceil(hi / 128) - floor(lo / 128)) and the rows the runs before it hold
 * n_runs == 0 selects nothing: out_keys is all HM_NO_MATCH (the _exchange entry needs n_runs >= 1; a rank without
 * selected rows joins the exchange through hm_exchange_merge with HM_NO_MATCH keys).
 *
 * hm_knn2_resident_runs: over a prepared image (hm_prepare) -- the k-NN kernel walks the runs in place, one launch
 * (kind::i8: + the query expansion).  hm_knn2_resident_runs_exchange: the same with the exchange of
 * hm_knn2_resident_exchange.  hm_knn2_runs: over packed rows -- the selected rows are gathered into the workspace
 * (36 bytes per selected row), hm_knn2 runs over them, and one small kernel maps the keys back.
 * hm_runs_workspace_bytes: workspace of the resident entries (prepared != 0, variant I8 / F4 / AUTO) or of
 * hm_knn2_runs (prepared == 0, any variant); 0 for invalid runs.  Nothing is sized by unselected rows.
 * hm_describe_runs_launch: host arithmetic, no device needed -- the resident launch for this selection as text (as
 * hm_describe_launch) and, when pieces_host != NULL, the tile walk: pieces_host[v] = (split, physical tile, first row,
 * end row) of virtual tile v, rows clipped to the run.  Returns the number of virtual tiles, or an hm_status < 0. */
HM_API size_t hm_runs_workspace_bytes(int64_t nq, const int64_t* runs_host, int64_t n_runs, int prepared, int variant);
HM_API int hm_describe_runs_launch(int64_t nq, int64_t nt, const int64_t* runs_host, int64_t n_runs, int variant,
                                   char* buf, size_t buf_bytes, int64_t* pieces_host);
HM_API int hm_knn2_resident_runs(const uint8_t* query, int64_t nq, int64_t q_stride, const void* train_prepared,
                                 int64_t nt, const int64_t* runs_host, const int64_t* runs_dev, int64_t n_runs,
                                 uint64_t train_base, uint64_t* out_keys, int variant, void* workspace,
                                 size_t workspace_bytes, void* stream);
HM_API int hm_knn2_resident_runs_exchange(const uint8_t* query, int64_t nq, int64_t q_stride, const void* train_prepared,
                                          int64_t nt, const int64_t* runs_host, const int64_t* runs_dev, int64_t n_runs,
                                          uint64_t train_base, int world, int rank, void* const* peer_buffers_host,
                                          int64_t max_rows, uint32_t epoch, uint64_t* out_keys, int variant,
                                          void* workspace, size_t workspace_bytes, void* stream);
HM_API int hm_knn2_runs(const uint8_t* query, int64_t nq, int64_t q_stride, const uint8_t* train, int64_t nt,
                        int64_t t_stride, const int64_t* runs_host, const int64_t* runs_dev, int64_t n_runs,
                        uint64_t train_base, uint64_t* out_keys, int variant, void* workspace, size_t workspace_bytes,
                        void* stream);

/* ---- tensor-core operand preparation (resident keyframe database) ---------------------
 * `variant` selects the operand format: HM_VARIANT_I8, HM_VARIANT_F4, or HM_VARIANT_AUTO = the
 * default tensor-core core (hm_default_tensor_variant()).  A prepared image must be consumed with the
 * variant it was prepared for. */
HM_API int hm_default_tensor_variant(void);
/* bytes of the prepared (+/-1, tiled, 128B-swizzled) image of n descriptors */
HM_API size_t hm_prepared_bytes(int64_t n, int variant);
/* expand n packed descriptors into `prepared` (hm_prepared_bytes(n, variant) bytes) */
HM_API int hm_prepare(const uint8_t* bits, int64_t n, int64_t stride, void* prepared, int variant, void* stream);
/* scratch bytes hm_knn2_prepared / hm_knn2_prepared_partials need (no operand expansion inside) */
HM_API size_t hm_prepared_workspace_bytes(int64_t nq, int64_t nt, int variant);
/* k-NN over operands prepared once (train side of a keyframe database stays resident) */
HM_API int hm_knn2_prepared(const void* query_prepared, int64_t nq,
                            const void* train_prepared, int64_t nt,
                            uint64_t train_base, uint64_t* out_keys, int variant,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Same k-NN, but the per-train-split partial keys are left unmerged in the workspace:
 * *out_partials -> [*out_groups][nq][2] (valid until the workspace is reused on the stream).
 * Feed them to hm_exchange_merge (or hm_merge_top2) to save one launch on the sharded path. */
HM_API int hm_knn2_prepared_partials(const void* query_prepared, int64_t nq,
                                     const void* train_prepared, int64_t nt, uint64_t train_base, int variant,
                                     void* workspace, size_t workspace_bytes, void* stream,
                                     const uint64_t** out_partials, int* out_groups);

/* ---- epilogues ------------------------------------------------------------------------ */
/* keys[groups][rows][2] -> out_keys[rows][2]: the 2 smallest of the 2*groups candidates per row.
 * Merges per-shard results after the all-gather of the sharded keyframe database. */
HM_API int hm_merge_top2(const uint64_t* keys, int groups, int64_t rows, uint64_t* out_keys, void* stream);

/* Fused exchange + merge for the sharded keyframe database (one launch per rank, no NCCL call):
 * every rank pushes its [rows][2] local keys straight into slot `rank` of every peer's symmetric
 * buffer with NVLink peer stores, publishes a per-CTA epoch flag (release, system scope), waits for
 * the matching flags of all peers (acquire), and merges the `world` slots into out_keys.
 *  peer_buffers_host[world]  host array of DEVICE pointers to the same symmetric allocation on each
 *                            rank (peer-mapped, e.g. torch.distributed._symmetric_memory buffer_ptrs);
 *                            each at least hm_exchange_bytes(max_rows, world) bytes, zero-initialised
 *  epoch                     strictly increasing per call (1, 2, 3, ...), identical on all ranks
 *  local_keys[local_groups][rows][2]  this rank's candidates; local_groups > 1 folds the merge of the
 *                            k-NN kernel's train splits (hm_knn2_prepared_partials) into the same launch
 * All ranks must launch the call; the kernels wait on one another across GPUs (never run two ranks
 * on one GPU).  A peer that never arrives trips a bounded spin and the kernel traps. */
HM_API size_t hm_exchange_bytes(int64_t max_rows, int world);
HM_API int hm_exchange_merge(const uint64_t* local_keys, int local_groups, int64_t rows, int world, int rank,
                             void* const* peer_buffers_host, int64_t max_rows, uint32_t epoch,
                             uint64_t* out_keys, void* stream);

/* k-NN over prepared operands with the exchange folded into the same launch: the CTA that finishes a
 * query block last merges the train splits, pushes the block's keys to every peer, waits for the peers'
 * blocks and writes the globally merged top-2 -- compute + collective in ONE kernel per rank.
 * Same buffer / epoch contract as hm_exchange_merge (the two may be mixed on one buffer). */
HM_API int hm_knn2_prepared_exchange(const void* query_prepared, int64_t nq,
                                     const void* train_prepared, int64_t nt, uint64_t train_base,
                                     int world, int rank, void* const* peer_buffers_host, int64_t max_rows,
                                     uint32_t epoch, uint64_t* out_keys, int variant,
                                     void* workspace, size_t workspace_bytes, void* stream);

/* Ratio test / mutual check / reference distance filter + ordered compaction, per problem.
 *  fwd_keys[batch][nq][2]  from hm_knn2*(query, train)
 *  bwd_keys[batch][nt][2]  from hm_knn2*(train, query) (roles swapped); only read with HM_FLAG_MUTUAL
 *  ratio_lut_host[257]     host pointer, lut[d2] = ceil(ratio * d2) in float64; only with HM_FLAG_RATIO
 *  out_q/out_t/out_d[batch][nq] int32, ordered by queryIdx; out_count[batch]
 */
HM_API int hm_filter_matches(const uint64_t* fwd_keys, int64_t nq, const uint64_t* bwd_keys, int64_t nt,
                             int batch, unsigned flags, const uint16_t* ratio_lut_host, double dist_threshold,
                             int32_t* out_q, int32_t* out_t, int32_t* out_d, int32_t* out_count,
                             void* stream);

/* ---- keyframe database: Lowe ratio test + database-wide mutual check over the global top-2 ---------------------
 * keys[nq][2] are the GLOBAL top-2 keys of a query batch over the whole (possibly sharded) database, as
 * hm_knn2_resident / hm_merge_top2 / the fused exchange return them (trainIdx = global row).
 *
 * hm_db_mutual_flags: the mutual check for ONE shard, the rows [row_lo, row_lo + shard_rows) held packed in
 * shard_bits (shard_rows rows, t_stride bytes apart).  For every query q whose best row t1 = keys[q][0] lies in this
 * range (and, with HM_FLAG_RATIO, that passes the ratio test), the nearest query of row t1 over all nq rows of `query`
 * is computed (lowest query index on ties); out_flags[q] = 1 iff that is q.  Every other entry of out_flags[nq] is
 * written 0, including queries whose t1 another shard owns, so the element-wise MAX over the shards' flags is the
 * database-wide answer.  Work is a top-1 k-NN of at most nq gathered shard rows against the nq queries; with the
 * kind::mxf4 core (HM_VARIANT_F4, or AUTO when it resolves to it for nq x nq) only the rows this shard owns are
 * computed, the count of which stays on the device.  Nothing is proportional to the database size: the workspace is
 * hm_db_mutual_workspace_bytes(nq, variant).  flags: HM_FLAG_RATIO and HM_FLAG_MUTUAL only.  Unlike every other
 * workspace, this one must be 256-byte aligned (the base of a cudaMalloc or torch allocation is): a workspace that is
 * NULL, smaller, or not 256-byte aligned is HM_ERR_WORKSPACE.
 *
 * hm_db_filter: ratio test (HM_FLAG_RATIO) and mutual check (HM_FLAG_MUTUAL: keep q iff mutual_flags[q] != 0) on the
 * global keys, then the ordered compaction: out_q / out_t / out_d[nq] (queryIdx, global row, distance) ordered by
 * queryIdx, *out_count matches.  mutual_flags may be NULL only without HM_FLAG_MUTUAL; with neither flag every query
 * keeps its best row (knnMatch k=1). */
HM_API size_t hm_db_mutual_workspace_bytes(int64_t nq, int variant);
HM_API int hm_db_mutual_flags(const uint64_t* keys, int64_t nq, const uint8_t* query, int64_t q_stride,
                              const uint8_t* shard_bits, int64_t shard_rows, int64_t t_stride, uint64_t row_lo,
                              unsigned flags, const uint16_t* ratio_lut_host, uint8_t* out_flags,
                              int variant, void* workspace, size_t workspace_bytes, void* stream);
HM_API int hm_db_filter(const uint64_t* keys, int64_t nq, const uint8_t* mutual_flags, unsigned flags,
                        const uint16_t* ratio_lut_host, int32_t* out_q, int32_t* out_t, int32_t* out_d,
                        int32_t* out_count, void* stream);

/* knn2 (+ the swapped pass when HM_FLAG_MUTUAL) + hm_filter_matches in one enqueue.
 * out_keys (fwd, [batch][nq][2]) may be NULL when the caller only wants the match list.
 * With the kind::mxf4 core the forward k-NN kernel applies the ratio test to each row's final keys itself and marks the
 * best train row of every survivor as a candidate; the swapped pass then runs over the candidate train rows only
 * (gathered in-kernel from a device-side list, row count read on the device: nothing is synchronised with the host).
 * Same result as the full swapped pass; the workspace of hm_workspace_bytes() includes the candidate tables. */
HM_API int hm_match_fused(const uint8_t* query, int64_t nq, int64_t q_stride, int64_t q_batch_stride,
                          const uint8_t* train, int64_t nt, int64_t t_stride, int64_t t_batch_stride,
                          int batch, unsigned flags, const uint16_t* ratio_lut_host, double dist_threshold,
                          int32_t* out_q, int32_t* out_t, int32_t* out_d, int32_t* out_count,
                          uint64_t* out_keys,
                          int variant, void* workspace, size_t workspace_bytes, void* stream);

/* ---- consumer of the match list: replaces the two list-building loops of
 *      /root/reference/utils.py:13-19 (pose_estimation_2d2d) and :41-47 (triangulation) ------------- */
/* For every problem b and every match m < count[b] of a match list (q_idx / t_idx / count as written by
 * hm_filter_matches / hm_match_fused, `stride` = elements per problem = its nq):
 *     out_query_pts[b][m] = query_pts[b][q_idx[b][m]]     (current frame, features[m.queryIdx].position)
 *     out_train_pts[b][m] = train_pts[b][t_idx[b][m]]     (last frame,    features[m.trainIdx].position)
 * Points are (x, y) int32 pairs, 8-byte aligned; entries at m >= count[b] are left untouched. */
HM_API int hm_gather_points(const int32_t* q_idx, const int32_t* t_idx, const int32_t* count, int64_t stride, int batch,
                            const int32_t* query_pts, int64_t nq, const int32_t* train_pts, int64_t nt,
                            int32_t* out_query_pts, int32_t* out_train_pts, void* stream);

/* ---- detection mask: replaces /root/reference/utils.py:58-74 (get_featured_detection_mask) ----------
 * mask[h][w] (uint8, rows `row_stride` bytes apart) = inner ? 0 : 255 everywhere, then for each of the n
 * points (x, y int32 pairs, 8-byte aligned) the filled rectangle [x-radius, x+radius] x [y-radius, y+radius]
 * (inclusive, clipped to the image, like cv2.rectangle(..., cv2.FILLED)) = inner ? 255 : 0. */
HM_API int hm_rasterize_mask(const int32_t* points, int64_t n, int radius, int inner,
                             uint8_t* mask, int h, int w, int64_t row_stride, void* stream);

/* ---- host-buffer convenience (what a non-torch caller binds) --------------------------- */
typedef struct hm_context hm_context; /* owns a stream, device scratch, pinned staging, frame slots and a small
                                         cache of CUDA graphs; one context per calling thread (not thread-safe) */
HM_API int hm_context_create(hm_context** out_ctx);
HM_API void hm_context_destroy(hm_context* ctx);
/* numpy-in / numpy-out twin of hm_knn2: H2D, kernels, D2H, synchronises before returning */
HM_API int hm_knn2_host(hm_context* ctx, const uint8_t* query_host, int64_t nq,
                        const uint8_t* train_host, int64_t nt, uint64_t* out_keys_host, int variant);

/* Host-buffer query of a resident prepared database (the keyframe-database step, numpy in / keys out): pinned staging
 * and H2D of the packed query, hm_knn2_resident (world <= 1) or hm_knn2_resident_exchange, D2H of the keys, all on the
 * context's stream.  _begin only enqueues -- the caller may allocate its result objects while the kernel runs -- and
 * _end synchronises and copies the nq x 2 keys out.  One query in flight per context.  The database must have been
 * prepared before the call (synchronise the stream that ran hm_prepare). */
HM_API int hm_resident_query_begin(hm_context* ctx, const uint8_t* query_host, int64_t nq, int64_t q_stride,
                                   const void* train_prepared, int64_t nt, uint64_t train_base, int variant,
                                   int world, int rank, void* const* peer_buffers_host, int64_t max_rows,
                                   uint32_t epoch);
HM_API int hm_resident_query_end(hm_context* ctx, int64_t nq, uint64_t* out_keys_host);

/* numpy-in / numpy-out twin of hm_match_fused (batch = 1): H2D of both descriptor sets through
 * pinned staging, k-NN (+ swapped pass with HM_FLAG_MUTUAL), filter, D2H, one synchronisation.
 * out_q/out_t/out_d_host[nq] int32, *out_count_host = number of matches (ordered by queryIdx).
 * This is the call behind BruteForceFeatureMatcher.match() for numpy inputs. */
HM_API int hm_match_host(hm_context* ctx, const uint8_t* query_host, int64_t nq, int64_t q_stride,
                         const uint8_t* train_host, int64_t nt, int64_t t_stride,
                         unsigned flags, const uint16_t* ratio_lut_host, double dist_threshold, int variant,
                         int32_t* out_q_host, int32_t* out_t_host, int32_t* out_d_host, int32_t* out_count_host);

/* ---- resident frames (SURVEY.md 8f ranks 1 + 2): replaces the per-call repacking of
 *      /root/reference/primitives.py:200-205 + frontend.py:181-187 and the point loops of utils.py:13-19 ---- */
/* problems up to this size take the single-launch path of hm_match_host / hm_frame_match (csrc/hm_small.cu) */
#define HM_SMALL_MAX_ROWS 1024
#define HM_SMALL_MAX_PAIRS 262144
#define HM_FRAME_SLOTS 16
/* Upload a frame ONCE into `slot` (0 .. HM_FRAME_SLOTS-1) of the context: n descriptors (rows `stride` bytes
 * apart) and, when points_host != NULL, its n keypoint positions (x, y int32 pairs).  Asynchronous; later
 * calls on the context are ordered after it. */
HM_API int hm_frame_put(hm_context* ctx, int slot, const uint8_t* desc_host, int64_t n, int64_t stride,
                        const int32_t* points_host);
/* ---- ORB descriptor stage on the device: replaces the descriptor half of
 *      /root/reference/feature_detectors.py:25-26 (cv2.ORB.detectAndCompute), called from
 *      /root/reference/frontend.py:245-249.  Keypoint DETECTION stays with cv2 on the host; what runs here is what
 *      cv2 does after it: gray conversion, the 1.2^level scale pyramid (bit-exact bilinear, each level from the
 *      previous one), the 32-pixel reflect-101 frame, the 7 x 7 sigma-2 blur and the 256 rotated rBRIEF comparisons
 *      (oracle/orb_oracle.py states every step; results are bit-identical to cv2 4.13 for the same keypoints). */
#define HM_ORB_MAX_LEVELS 16
#define HM_ORB_BORDER 32
/* A geometry (rows, cols, n_levels) is accepted when 1 <= n_levels <= HM_ORB_MAX_LEVELS, each side is at most 16384 and
 * every level 0 .. n_levels-1 is more than HM_ORB_BORDER pixels on both sides (the reflected frame fits inside it).
 * Otherwise hm_orb_workspace_bytes returns 0 and the calls below return HM_ERR_INVALID_ARGUMENT. */
HM_API size_t hm_orb_workspace_bytes(int rows, int cols, int n_levels);
/* size and 1 / scale of pyramid level `level` (host arithmetic, no device needed) */
HM_API int hm_orb_level_geometry(int rows, int cols, int level, int* out_rows, int* out_cols, float* out_inv_scale);
/* (cos, sin) pairs of keypoint angles in degrees, with the arithmetic cv2 uses: float radians, double cos / sin, rounded to float (host) */
HM_API int hm_orb_angles_to_cs(const float* angle_deg_host, int64_t n, float* cs_host);
/* image: device uint8, 1 (gray) or 3 (BGR) channels, rows `row_stride` bytes apart -> blurred pyramid in `workspace` */
HM_API int hm_orb_build_pyramid(const uint8_t* image, int rows, int cols, int64_t row_stride, int channels, int n_levels,
                                void* workspace, size_t workspace_bytes, void* stream);
/* n keypoints: kp_xy = KeyPoint.pt (level-0 pixels, float pairs, 8-byte aligned), kp_cs = hm_orb_angles_to_cs of
 * KeyPoint.angle, kp_octave = KeyPoint.octave (< n_levels) -> out_desc[n] rows of 32 bytes, `out_stride` bytes apart.
 * `workspace` is the one hm_orb_build_pyramid filled for the same (rows, cols, n_levels).  Octaves are not checked here:
 * one outside 0 .. n_levels-1 is clamped to that range (hm_frame_put_orb rejects them). */
HM_API int hm_orb_describe(const void* workspace, int rows, int cols, int n_levels, const float* kp_xy, const float* kp_cs,
                           const int32_t* kp_octave, int64_t n, uint8_t* out_desc, int64_t out_stride, void* stream);
/* Host image + keypoints -> descriptors written straight into frame slot `slot` (they never visit the host unless
 * out_desc_host is non-NULL); points_host as in hm_frame_put.  One H2D, the kernels above, no synchronisation unless
 * a copy is requested. */
HM_API int hm_frame_put_orb(hm_context* ctx, int slot, const uint8_t* image_host, int rows, int cols, int64_t row_stride,
                            int channels, int n_levels, const float* kp_xy_host, const float* kp_angle_deg_host,
                            const int32_t* kp_octave_host, int64_t n, const int32_t* points_host, uint8_t* out_desc_host);

/* hm_match_host between two resident frames (query = current frame, train = last frame).  Outputs as
 * hm_match_host; out_q/out_t/out_d may be NULL.  When both out_*_pts_host are non-NULL (each [nq][2] int32)
 * they receive the matched keypoint positions, gathered on the device: [m] = position of the query / train
 * feature of match m -- the arrays utils.py:13-19 builds for cv2.findEssentialMat. */
HM_API int hm_frame_match(hm_context* ctx, int train_slot, int query_slot, unsigned flags,
                          const uint16_t* ratio_lut_host, double dist_threshold, int variant,
                          int32_t* out_q_host, int32_t* out_t_host, int32_t* out_d_host,
                          int32_t* out_query_pts_host, int32_t* out_train_pts_host, int32_t* out_count_host);

#ifdef __cplusplus
}
#endif
#endif /* HM_MATCHER_H_ */

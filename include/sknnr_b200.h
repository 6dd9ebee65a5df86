/* sknnr_b200 - C ABI of the B200-native query-time hot path of lemma-osu/sknnr.
 *
 * The reference (pure Python) has no FFI layer; its narrowest seams for this path are
 *
 *   S1  super().kneighbors(X=..., n_neighbors=..., return_distance=True)
 *       ref:src/sknnr/_base.py:162-164   (Z f64 [n_q,d'] | None, k) -> (dist f64, idx i64)
 *       followed by the re-ordering at :166-175
 *   S2  TransformedKNeighborsRegressor._transform_X       ref:src/sknnr/_base.py:236-239
 *   S3  regressor_.predict / regressor_.score             ref:src/sknnr/_base.py:346-352
 *
 * Each entry point below names the seam it replaces.  Plain pointers and sizes only, no
 * torch types; every function returns 0 on success or a negative SKNNR_E* code, never
 * throws, and leaves a thread-local message for sknnr_last_error().  There is no CPU
 * fallback anywhere behind this ABI: without a CUDA device every compute call fails.
 *
 * Ownership: the caller owns every input/output buffer; an index handle owns only device
 * copies of the fitted state plus its scratch and is a rebuildable cache.  A handle is
 * internally locked, so concurrent calls on one handle serialise; distinct handles are
 * independent.
 */
#ifndef SKNNR_B200_H
#define SKNNR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SKNNR_ABI_VERSION 1

/* error codes */
#define SKNNR_OK 0
#define SKNNR_EINVAL (-1)   /* bad argument (the Python layer validates first)        */
#define SKNNR_ECUDA (-2)    /* CUDA runtime / launch failure                           */
#define SKNNR_ENODEV (-3)   /* no CUDA device                                          */
#define SKNNR_ENOMEM (-4)   /* device or pinned-host allocation failed                 */
#define SKNNR_EUNSUP (-5)   /* shape outside what the kernels cover                    */
#define SKNNR_ENONFINITE (-6) /* SKNNR_CHECK_FINITE: a query value is NaN or +-inf      */

/* dtype of a query matrix */
#define SKNNR_F64 0
#define SKNNR_F32 1

/* flags for the query calls */
#define SKNNR_EXCLUDE_SELF 1u   /* X=None semantics: search k+1, drop the query itself
                                   ($SP/sklearn/neighbors/_base.py:821-826,929-958), used by
                                   IndependentPredictorMixin (ref:src/sknnr/_base.py:37-40)  */
#define SKNNR_DETERMINISTIC 2u  /* use_deterministic_ordering (ref:src/sknnr/_base.py:166-175) */
#define SKNNR_TRANSFORMED 4u    /* X is already in the estimator's space (seam S1 alone,
                                   RawKNNRegressor); otherwise S2 is fused in front         */
#define SKNNR_DEVICE_PTRS 8u    /* X and all outputs are device pointers on the handle's
                                   device; work is enqueued on `stream` and NOT synchronised */

#define SKNNR_CHECK_FINITE 16u  /* host-buffer calls: fail with SKNNR_ENONFINITE when a query value
                                   is NaN / +-inf (the projection kernel reads every value anyway;
                                   replaces the host pass of sklearn's validate_data,
                                   $SP/sklearn/neighbors/_base.py:831-838); outputs are undefined then */

/* prediction weights (seam S3, $SP/sklearn/neighbors/_base.py:74-117) */
#define SKNNR_W_NONE 0      /* no prediction requested                                    */
#define SKNNR_W_UNIFORM 1   /* mean of the k targets                                       */
#define SKNNR_W_DISTANCE 2  /* 1/d, rows containing d==0 use the (d==0) indicator          */

/* search engines (diagnostics / benchmarking; 0 lets the library choose) */
#define SKNNR_ENGINE_AUTO 0
#define SKNNR_ENGINE_SIMT 1     /* FP32 FFMA2 register-tiled kernel                        */
#define SKNNR_ENGINE_TENSOR 2   /* tcgen05 TF32 filter kernel                              */
#define SKNNR_ENGINE_EXACT 3    /* FP64 exhaustive kernel (the certificate's fallback)     */

typedef struct sknnr_index sknnr_index;           /* Euclidean-space estimators */
typedef struct sknnr_hamming_index sknnr_hamming_index; /* RFNN node-ID estimators    */
typedef struct sknnr_forest sknnr_forest;               /* fitted forests of an RFNodeTransformer */

/* counters of the last query call on a handle (all int64) */
typedef struct sknnr_stats {
    int64_t n_queries;       /* rows processed                                           */
    int64_t n_fallback;      /* rows whose certificate failed and were re-searched exactly */
    int64_t kernel_launches; /* kernels of this library launched by the call              */
    int64_t h2d_bytes;       /* bytes copied host->device by the call                     */
    int64_t d2h_bytes;       /* bytes copied device->host by the call                     */
    int64_t engine;          /* SKNNR_ENGINE_* actually used                              */
    double search_ms;        /* device time of the dominant (search) kernels, CUDA events;
                                only filled when sknnr_set_option("timing", 1)            */
} sknnr_stats;

const char *sknnr_last_error(void);
int sknnr_abi_version(void);
int sknnr_device_count(int *count);

/* Global knobs (environment-style; never estimator constructor arguments):
 *   "engine"      SKNNR_ENGINE_*           (default AUTO)
 *   "chunk_rows"  rows per internal chunk  (default 1<<20; device-pointer calls use twice that)
 *   "host_slots"  1..8: a host-buffer call keeps min(4, value) chunks in flight (default 8)
 *   "timing"      0/1 record search_ms     (default 0)
 *   "kc"          0/8/16/32 minimum length of the FP32 (SIMT) search's candidate list (default 16);
 *                 0 picks the smallest list that holds k+1 (longer lists = fewer certificate
 *                 failures, more insertions)
 *   "tc_streams"  0/1/2 candidate streams per query of the tensor engine (default 0 = two
 *                 streams of 8 while k (+1) <= 8, else one of 16)
 *   "tc_seed_stride" 0..64: the tensor engine pre-scans one reference tile in n to seed its
 *                 thresholds (default 4; 0 = the default too: the engine never starts cold, and
 *                 reference sets below 192 / 64 tiles are pre-scanned at stride <= 2 / 1)
 *   "stage_rows"  rows per chunk of a call with pageable buffers (default 1<<19)
 *   "tc_debug"    timing experiments only (bit 0 skips the hit path, bit 2 skips the tile
 *                 loads: results are wrong)                                             */
int sknnr_set_option(const char *name, int64_t value);

/* The chunk schedule a host-buffer call of n_q rows uses with chunks of chunk_rows (host code only, no
 * device needed): rows_out[0 .. min(cap, *n_chunks)) = rows per chunk.  From four chunks' worth of rows
 * up the schedule ramps up (1/4, 1/2, 1, ...) and down (..., 1/2, 1/4): the first chunk's copy in and
 * the last chunk's copy out overlap no kernel. */
int sknnr_host_chunk_plan(int64_t n_q, int64_t chunk_rows, int64_t *rows_out, int32_t cap, int32_t *n_chunks);

/* ---- Euclidean-space index: Raw / Euclidean / Mahalanobis / MSN / GNN ------------------
 * Fitted state of one estimator.  The four float transformers are one affine map
 *     Z = ((X - center) / scale) @ proj
 * (StandardScalerWithDOF: $SP/sklearn/preprocessing/_data.py:1131-1134 with scale_ from
 *  ref:src/sknnr/transformers/_base.py:66; MahalanobisTransformer
 *  ref:src/sknnr/transformers/_mahalanobis_transformer.py:55; CCorATransformer
 *  ref:src/sknnr/transformers/_ccora_transformer.py:70; CCATransformer
 *  ref:src/sknnr/transformers/_cca_transformer.py:87).
 *
 *   fit_z   [n_ref, d_out] f64 C-order  - regressor_._fit_X (transformed reference plots)
 *   center  [d_in] or NULL (no centring); scale [d_in] or NULL (no scaling)
 *   proj    [d_in, d_out] f64 C-order or NULL (identity, d_in == d_out)
 *   y       [n_ref, n_out] f64 C-order or NULL (kneighbors only); regressor_._y
 * All pointers are HOST pointers; the data is copied.                                    */
int sknnr_index_create(const double *fit_z, int64_t n_ref, int32_t d_out,
                       const double *center, const double *scale, const double *proj,
                       int32_t d_in, const double *y, int32_t n_out, int32_t device,
                       sknnr_index **out);
int sknnr_index_destroy(sknnr_index *index);

/* kneighbors (+ optional predict) for n_q query rows.  Replaces S2+S1(+S3) in one call.
 *
 *   X          [n_q, d_in] (or [n_q, d_out] with SKNNR_TRANSFORMED), dtype x_dtype,
 *              row stride ldx elements.  With SKNNR_EXCLUDE_SELF X must be NULL: the query
 *              set is the reference set itself and n_q is ignored (= n_ref).
 *   row_offset global row number of X[0] - the |idx - query_row| tie-break key
 *              (ref:src/sknnr/_base.py:171) of a sharded caller.
 *   k          neighbours returned per row (1 <= k; k + exclude_self <= min(n_ref, 32)).
 *   decimals   RawKNNRegressor.DISTANCE_PRECISION_DECIMALS (ref:src/sknnr/_base.py:102).
 *   out_dist   [n_q, k] f64 or NULL;  out_idx [n_q, k] i64 or NULL
 *   weights    SKNNR_W_*; out_pred [n_q, n_out] f64 (required unless SKNNR_W_NONE)
 *   stream     cudaStream_t as void* (only with SKNNR_DEVICE_PTRS; else ignored)
 * Without SKNNR_DEVICE_PTRS the call is synchronous and every pointer may be a pageable host,
 * page-locked host or device pointer (unified addressing; a peer GPU's memory mapped with
 * sknnr_ipc_open included): device-resident X is read in place, results bound for device memory
 * leave each chunk as one copy-engine transfer.                                               */
int sknnr_kneighbors(sknnr_index *index, const void *X, int32_t x_dtype, int64_t n_q,
                     int64_t ldx, int64_t row_offset, int32_t k, uint32_t flags,
                     int32_t decimals, double *out_dist, int64_t *out_idx, int32_t weights,
                     double *out_pred, void *stream);

/* S2 alone: Z = ((X - center) / scale) @ proj, out_z [n_q, d_out] f64 (host pointers).    */
int sknnr_transform(sknnr_index *index, const void *X, int32_t x_dtype, int64_t n_q,
                    int64_t ldx, double *out_z);

/* S3 with caller-supplied weights (callable `weights=` evaluated by Python on the
 * distances): out_pred[i, :] = sum_c w[i,c] * y[idx[i,c], :] / sum_c w[i,c]
 * ($SP/sklearn/neighbors/_regression.py:262-267).  Host pointers.                         */
int sknnr_weighted_average(sknnr_index *index, const int64_t *idx, const double *w,
                           int64_t n_q, int32_t k, double *out_pred);

int sknnr_index_stats(sknnr_index *index, sknnr_stats *out);
/* Rows of the last call that left each stage of the engine cascade uncertified:
 * out3[0] after the tensor engine's first pass (= stats.n_fallback), out3[1] rows that reached the
 * FP32 engine, out3[2] rows that reached the exhaustive float64 kernel.                      */
int sknnr_index_cascade_counts(sknnr_index *index, int64_t *out3);

/* ---- Hamming index: RFNNRegressor (metric="hamming" over terminal-node IDs) -------------
 * Replaces sklearn's brute Hamming branch + scipy cdist_hamming
 * ($SP/sklearn/neighbors/_base.py:879-908,715-754; $SP/scipy/spatial/distance.py:1718-1723)
 * reached with w = hamming_weights_ (ref:src/sknnr/_weighted_trees.py:65-98,139-140).
 *
 *   ref_codes [n_ref, n_trees] u16 C-order: per-tree node codes.  Only equality matters, so
 *             the host maps each tree's node IDs (int64 from
 *             ref:src/sknnr/transformers/_tree_node_transformer.py:177-201) to dense codes
 *             in [0, 31743]; 31743 is reserved for "matches nothing".
 *   w         [n_trees] f64 hamming weights.  Equal weights (RFNNRegressor) use the integer
 *             kernel and a host-built table of the float64 distances reachable (bit-exact with
 *             SciPy's left-to-right sums).  Unequal weights (GBNNRegressor's tree weights,
 *             ref:src/sknnr/transformers/_gbnode_transformer.py:288-310; user forest_weights)
 *             run a 16-bit fixed-point filter, recompute the survivors in float64 in SciPy's
 *             order and certify the top k; uncertified rows, negative weights and k > 24 use
 *             the exhaustive float64 kernel.  Results are bit-equal in every case.
 *   y         [n_ref, n_out] f64 or NULL.                                                  */
int sknnr_hamming_index_create(const uint16_t *ref_codes, int64_t n_ref, int32_t n_trees,
                               const double *w, const double *y, int32_t n_out,
                               int32_t device, sknnr_hamming_index **out);
int sknnr_hamming_index_destroy(sknnr_hamming_index *index);

/* Same contract as sknnr_kneighbors; q_codes [n_q, n_trees] u16, row stride ldq elements.
 * Neighbours are the k smallest by (distance, index): the lowest index wins every tie.     */
int sknnr_hamming_kneighbors(sknnr_hamming_index *index, const uint16_t *q_codes,
                             int64_t n_q, int64_t ldq, int64_t row_offset, int32_t k,
                             uint32_t flags, int32_t decimals, double *out_dist,
                             int64_t *out_idx, int32_t weights, double *out_pred,
                             void *stream);
int sknnr_hamming_weighted_average(sknnr_hamming_index *index, const int64_t *idx,
                                   const double *w, int64_t n_q, int32_t k,
                                   double *out_pred);
int sknnr_hamming_index_stats(sknnr_hamming_index *index, sknnr_stats *out);

/* ---- Forests: RFNodeTransformer.transform on the device (scope row f1) -------------------
 * Replaces ref:src/sknnr/transformers/_tree_node_transformer.py:177-201 (est.apply per forest,
 * hstack) -> $SP/sklearn/tree/_tree.pyx:977-994 (Tree._apply_dense): X is cast to float32, an
 * internal node sends a row left iff (double)x[feature] <= threshold, NaN follows
 * missing_go_to_left, a node with children_left == -1 is a leaf.
 *
 * All trees of all forests are concatenated in transform's column order:
 *   tree_offsets [n_trees + 1] first node of every tree in the arrays below
 *   children_left / children_right / feature / threshold / missing_go_to_left [n_nodes]:
 *             scikit-learn's tree_ arrays (child indices local to their tree, -1 = leaf;
 *             missing_go_to_left may be NULL)
 *   node_code [n_nodes] u16 or NULL: the node code the Hamming index uses for each (leaf)
 *             node, 31743 = "matches nothing"; NULL = the node ID itself                    */
int sknnr_forest_create(const int32_t *tree_offsets, const int32_t *children_left,
                        const int32_t *children_right, const int32_t *feature,
                        const double *threshold, const uint8_t *missing_go_to_left,
                        const uint16_t *node_code, int32_t n_trees, int32_t n_features,
                        int32_t device, sknnr_forest **out);
int sknnr_forest_destroy(sknnr_forest *forest);
/* Node IDs (per tree, as est.apply returns them) of host rows X [n_q, >= n_features]. */
int sknnr_forest_apply(sknnr_forest *forest, const void *X, int32_t x_dtype, int64_t n_q,
                       int64_t ldx, int32_t *out_ids);
/* sknnr_hamming_kneighbors on raw feature rows: forest walk -> node codes -> Hamming search
 * without leaving the device.  X [n_q, ldx] of x_dtype (host, or device with
 * SKNNR_DEVICE_PTRS); every other argument as in sknnr_hamming_kneighbors.                  */
int sknnr_hamming_kneighbors_forest(sknnr_hamming_index *index, sknnr_forest *forest,
                                    const void *X, int32_t x_dtype, int64_t n_q, int64_t ldx,
                                    int64_t row_offset, int32_t k, uint32_t flags,
                                    int32_t decimals, double *out_dist, int64_t *out_idx,
                                    int32_t weights, double *out_pred, void *stream);

/* ---- Raster front end (scope row f4) -----------------------------------------------------
 * The caller either side of the path when the queries are the pixels of a map (the
 * "sknnr-spatial"-style loop around est.kneighbors / est.predict, ref:src/sknnr/_base.py:285-352):
 * flatten a band-major image to [n_pix, d], drop masked pixels, query, write band-major layers.
 * Here the image block goes to the device as it is and the transpose, the mask, the compaction
 * and the scatter back run next to the search.
 *
 *   bands      host, band b = bands + b * band_stride elements of x_dtype, n_pix pixels each
 *              (index->d_in bands, raw feature space)
 *   a pixel is masked when any band is NaN / +-inf, or equals `nodata` while use_nodata != 0
 *   the unmasked pixels, in pixel order, are the query rows 0 .. n_valid-1 of one
 *   sknnr_kneighbors call (that numbering feeds the deterministic ordering key)
 *   out_dist / out_idx [k][n_pix], out_pred [n_out][n_pix]: band-major layers (any may be NULL as
 *              in sknnr_kneighbors); masked pixels receive fill_dist / fill_idx / fill_pred
 *   flags      SKNNR_DETERMINISTIC or 0;  n_valid (may be NULL) <- number of unmasked pixels  */
int sknnr_raster_kneighbors(sknnr_index *index, const void *bands, int32_t x_dtype, int64_t n_pix,
                            int64_t band_stride, int32_t use_nodata, double nodata, int32_t k,
                            uint32_t flags, int32_t decimals, double *out_dist, int64_t *out_idx,
                            int32_t weights, double *out_pred, double fill_dist, int64_t fill_idx,
                            double fill_pred, int64_t *n_valid);

/* The same for the tree-node estimators (RFNN / GBNN): the unmasked pixels' feature rows are walked
 * through `forest` on the device and searched in the Hamming index (forest->n_features bands).  */
int sknnr_hamming_raster_kneighbors_forest(sknnr_hamming_index *index, sknnr_forest *forest,
                                           const void *bands, int32_t x_dtype, int64_t n_pix,
                                           int64_t band_stride, int32_t use_nodata, double nodata,
                                           int32_t k, uint32_t flags, int32_t decimals,
                                           double *out_dist, int64_t *out_idx, int32_t weights,
                                           double *out_pred, double fill_dist, int64_t fill_idx,
                                           double fill_pred, int64_t *n_valid);

/* Pinned host memory for callers that stream large rasters (cudaHostAlloc / cudaFreeHost). */
int sknnr_host_alloc(void **ptr, int64_t bytes);
int sknnr_host_free(void *ptr);

/* Device buffers shared between the one-process-per-GPU ranks of a box (SURVEY.md section 8e: the
 * gather of (dist, idx, pred) to one rank).  The root rank allocates the full result arrays with
 * sknnr_device_alloc and exports them (64-byte CUDA IPC handle); every other rank opens them and
 * passes its slice as out_dist / out_idx / out_pred of a SKNNR_DEVICE_PTRS query, so the finishing
 * kernels store their rows straight into the root's memory over NVLink - the gather is fused into
 * the compute, no collective follows it.  sknnr_device_copy: kind 0 = device to device (async on
 * `stream`), 1 = host to device, 2 = device to host (both synchronous).                    */
int sknnr_device_alloc(int32_t device, void **ptr, int64_t bytes);
int sknnr_device_free(int32_t device, void *ptr);
int sknnr_ipc_export(int32_t device, void *ptr, void *handle64);
int sknnr_ipc_open(int32_t device, const void *handle64, void **ptr);
int sknnr_ipc_close(int32_t device, void *ptr);
int sknnr_device_copy(int32_t device, void *dst, const void *src, int64_t bytes, int32_t kind,
                      void *stream);

/* FP32 FMA-pipe peak probe: runs a register-resident FFMA2 loop on every SM and returns
 * the achieved TFLOP/s (the denominator of the SIMT roofline, measured not assumed).      */
int sknnr_measure_fp32_peak(int32_t device, double *tflops);

#ifdef __cplusplus
}
#endif
#endif /* SKNNR_B200_H */

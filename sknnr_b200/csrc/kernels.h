// Host-callable launchers of the sknnr_b200 kernels (internal; the public ABI is
// include/sknnr_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stddef.h>

namespace sk {

struct FinishParams;

// ---- element types of a query matrix / raster block: the x_dtype codes of include/sknnr_b200.h
// (SKNNR_F64 0, SKNNR_F32 1, SKNNR_U8 2, SKNNR_I16 3, SKNNR_U16 4, SKNNR_I32 5, SKNNR_I64 6) ------
// Bytes per element; 0 for an unknown code.
inline size_t x_dtype_size(int x_dtype) {
    switch (x_dtype) {
        case 0: case 6: return 8;
        case 1: case 5: return 4;
        case 3: case 4: return 2;
        case 2: return 1;
        default: return 0;
    }
}
// f(TX{}) with TX the element type of x_dtype (the kernel instantiation a launcher picks);
// cudaErrorInvalidValue for an unknown code
template <class F>
cudaError_t with_x_type(int x_dtype, F &&f) {
    switch (x_dtype) {
        case 0: return f(double{});
        case 1: return f(float{});
        case 2: return f(uint8_t{});
        case 3: return f(int16_t{});
        case 4: return f(uint16_t{});
        case 5: return f(int32_t{});
        case 6: return f(0LL);
        default: return cudaErrorInvalidValue;
    }
}

// ---- project.cu: Z = ((X - center) / scale) @ proj  (S2, a1-a4) -----------------------
// Writes Z as float64 rows (exact re-rank operand) and as the search kernel's query tile
// image [n_qtiles][dpad][256] f32 = -2 * (Z - mu).
// Also (optionally) the tensor-core engine's image [n_q/128][tc_kc][128][8] FP16 (two
// consecutive 128-row operands form one CTA tile of the tensor kernel), scaled by tc_sigma.
// Both images are zero-padded to a multiple of 1536 rows (padded_rows: every CTA tile size of
// either engine - 256, 384, 512 - divides it).  n_rows_dev != null makes
// the launch "compacted": only the first *n_rows_dev rows exist (device-side count).
inline long long padded_rows(long long n) { return (n + 1535) / 1536 * 1536; }
cudaError_t launch_project(const void *X, int x_dtype, long long ldx, long long n_q, int d_in,
                           int d_out, int dpad, const double *center, const double *scale,
                           const double *proj, const double *mu, double *z64, float *qimg,
                           __half *qimg_tc, int tc_kc, double tc_sigma, const int *n_rows_dev,
                           int *nonfinite, cudaStream_t st);
// z64c[i, :] = z64[list[i], :] for i < *count (rows whose certificate failed)
cudaError_t launch_gather_rows(const double *z64, int d, const int *list, const int *count,
                               long long max_rows, double *z64c, cudaStream_t st);

// ---- search_simt.cu --------------------------------------------------------------------
// distance of a float index (the values of SKNNR_METRIC_*)
constexpr int METRIC_L2 = 0;     // Euclidean
constexpr int METRIC_L1 = 1;     // Manhattan
constexpr int METRIC_LINF = 2;   // Chebyshev
size_t search_simt_smem_bytes(int dpad, int kc, int nstage);
int search_simt_pick_stages(int dpad, int kc);
cudaError_t launch_search_simt(const float *qimg, const float *rimg, int dpad, int n_rtiles,
                               long long n_q, int kc, int *cand_idx, float *cand_thr,
                               const int *n_rows_dev, int spread_ctas, int bypass_rows, cudaStream_t st,
                               int metric);
// n_rows_dev != null: compacted launch, the row count is read on the device; spread_ctas > 0 then
// deals the rows out over up to that many CTAs in units of one warp (0: one CTA per 384 rows); a compacted
// launch with fewer than bypass_rows rows does nothing (refine then hands the rows on, RefineArgs.bypass_rows)

// ---- search_tc.cu (tcgen05 / TMEM engine) ------------------------------------------------
// Two candidate-stream layouts: ns = 2 (two lists of up to 7 per query, k (+1) <= 7) and ns = 1 (one
// list of up to 15).  cand_idx is [n_q][16], cand_thr [n_q][ns]; every reference outside a query's
// lists has an approximate score >= the minimum of its ns thresholds.
size_t search_tc_smem_bytes(int kc_tot, int nstage, int ns, int cape);
int search_tc_pick_config(int kc_tot);   // ring stages | pending-queue depth << 8; 0: the shape does not fit
int search_tc_seed_tiles(int n_rtiles, int seed_stride);
extern int g_tc_debug;  // timing experiments: bit 0 = skip the hit path (wrong results)
// seed_stride: one reference tile in seed_stride is pre-scanned to seed the thresholds (0 = the
// default, 4; small reference sets use a denser stride, see search_tc_seed_stride)
cudaError_t launch_search_tc(const __half *qimg, const __half *rimg, int kc_tot, int n_rtiles,
                             long long n_q, int ns, int config, int seed_stride, int wide_joint, int *cand_idx,
                             float *cand_thr, const float *init_thr, const int *n_rows_dev, cudaStream_t st);
// wide_joint (two streams only): the joint threshold sits at rank 12 of the query's candidates instead of 10
// (fewer uncertified rows, more candidates to carry)
// init_thr != null: second pass - no seeding, row q starts from threshold init_thr[q]; n_rows_dev != null:
// compacted launch, the row count is read on the device

// ---- refine.cu -------------------------------------------------------------------------
struct RefineArgs {
    const double *z64;      // [n_q, d] queries in the estimator's space
    const double *ref64;    // [n_ref, d]
    const double *mu;       // [d] centroid used by the search images
    const int *cand_idx;    // [n_q, kc]
    const float *cand_thr;  // [n_q, n_thr]: a query's filter threshold is the minimum of its n_thr entries
    int n_thr;
    int kc;
    int d;
    long long n_q;
    int n_ref;
    double eps_s;           // relative error bound of the approximate score
    double r2max;           // max_j |ref_j - mu|^2
    double thr_scale;       // cand_thr holds thresholds of scores scaled by 1 / thr_scale (tensor engine: sigma^2)
    double qn_limit;        // rows with |q - mu|^2 >= qn_limit are never certified (FP16 range of the query image)
    int *fb_count;          // number of uncertified queries (device)
    int *fb_list;           // their row numbers (device, capacity n_q)
    float *fb_thr;          // null, or [capacity n_q]: per uncertified row, the score threshold under which a
                            // second pass of the same engine has to list every reference (retry_threshold)
    const int *n_rows_dev;  // compacted launch: only the first *n_rows_dev rows exist
    const int *row_map;     // compacted launch: row of the original chunk (goes into fb_list)
    int bypass_rows;        // compacted launch with fewer rows than this: the search was skipped, every row
                            // goes to fb_list unexamined
};
cudaError_t launch_refine(const RefineArgs &a, const FinishParams &fp, cudaStream_t st);
// The same stage for METRIC_L1 / METRIC_LINF: every candidate's float64 distance is recomputed in
// scikit-learn's order (sequential sum / max of |z_k - r_k|), so the distances are bit-equal to its
// own.  r2max holds max_j |ref_j - mu| in the metric's norm, qn_limit bounds |q - mu| the same way,
// thr_scale = 0.5 (the images hold -2 (x - mu)); compacted launches are not supported.
cudaError_t launch_refine_lp(const RefineArgs &a, int metric, const FinishParams &fp, cudaStream_t st);

// Exhaustive float64 search for the rows in list[0..*count) (or all rows when list==null):
// one CTA per row, all references, exact (distance, index) top-k, then finish_query.
struct ExactArgs {
    int metric;             // 0 = Euclidean (z64/ref64), 2 = Manhattan, 3 = Chebyshev; weighted Hamming
                            // (codes + w): 1 = uint16_t codes, 4 = uint32_t codes (wide mode)
    const double *z64;
    const double *ref64;
    int d;
    const void *qcodes;     // [n_q, ldq]
    const void *rcodes;     // [n_ref, n_trees]
    int n_trees;
    long long ldq;
    const double *w;        // [n_trees]
    double wsum;
    long long n_q;
    int n_ref;
    const int *list;
    const int *count;
    double *scratch;        // [grid, n_ref]
    double *big;            // [grid, 4 * (k + exclude_self)] - only read when k (+1) > 32
    int grid;
};
cudaError_t launch_exact(const ExactArgs &a, const FinishParams &fp, cudaStream_t st);

// S3 with caller weights
cudaError_t launch_weighted_average(const long long *idx, const double *w, long long n_q, int k,
                                    const double *y, int n_out, double *out_pred,
                                    cudaStream_t st);

// ---- hamming.cu ------------------------------------------------------------------------
constexpr int HAM_WC = 32;  // packed 32-bit words (= 64 trees) per staged chunk
// pack u16 codes [n, ldc] into tile images [n_tiles][n_chunks][HAM_WC][tile] u32
cudaError_t launch_hamming_pack(const uint16_t *codes, long long n, long long ldc, int n_trees,
                                int n_chunks, int tile, uint16_t pad_code, uint32_t *img,
                                cudaStream_t st);
// wq == null: equal weights, cand_cnt = mismatch counts.  wq [n_chunks * HAM_WC] (two 16-bit
// fixed-point weights per word): cand_cnt = fixed-point weight sums (kc 16 or 32 only)
cudaError_t launch_hamming_search(const uint32_t *qimg, const uint32_t *rimg, const uint32_t *wq,
                                  int n_chunks, int n_rtiles, long long n_q, int n_ref, int kc,
                                  int *cand_idx, int *cand_cnt, cudaStream_t st);
// mismatch counts -> float64 distances through the host-built table, then finish_query
cudaError_t launch_hamming_finish(const int *cand_idx, const int *cand_cnt, int kc,
                                  const double *lut, long long n_q, const FinishParams &fp,
                                  cudaStream_t st);
// Wide mode (trees with more than 31743 distinct node IDs): exact u32 codes, 0xFFFFFFFF = "matches
// nothing"; the 16-bit kernels above run as a filter on the hashed image of the codes.
constexpr uint32_t WIDE_NONE = 0xFFFFFFFFu;
__host__ __device__ inline uint16_t hamming_filter_code(uint32_t wide) {
    return wide == WIDE_NONE ? (uint16_t)31743 : (uint16_t)(wide % 31743u);
}
// codes [n, n_trees] <- filter codes of wide [n, ldw]
cudaError_t launch_hamming_hash(const uint32_t *wide, long long n, long long ldw, int n_trees, uint16_t *codes,
                                cudaStream_t st);
// exact (count or float64 distance) re-rank of the filter's candidates, certificate, finish_query or fb_list
struct HammingRefineArgs {
    const int *cand_idx;    // [n_q, kc]
    const int *cand_cnt;    // [n_q, kc] fixed-point weight sums, or hashed mismatch counts (lut != null)
    int kc;
    const void *qcodes;     // [n_q, ldq] exact codes: uint16_t, or uint32_t in wide mode
    long long ldq;
    const void *rcodes;     // [n_ref, n_trees] exact codes, the same type
    int n_trees;
    const double *lut;      // wide mode, equal weights: mismatch count -> float64 distance; null: unequal weights
    const double *w;        // [n_trees]
    double wsum;            // left-to-right float64 sum of w
    double scale, err;      // w_t = scale * wq_t + e_t, err >= sum |e_t| + float64 summation slack
    long long n_q;
    int *fb_count;
    int *fb_list;
};
// wide: the codes are uint32_t
cudaError_t launch_hamming_refine(const HammingRefineArgs &a, bool wide, const FinishParams &fp, cudaStream_t st);

// ---- forest.cu (RFNodeTransformer.transform on the device) -------------------------------
// One node of the flattened forests, 16 bytes (one LDG.128).  left < 0: leaf, `right` = the 16-bit
// node code the Hamming index uses for it.  feat: feature index, bit 31 set = missing values go left.
// thr = the largest float32 <= scikit-learn's float64 threshold: the walked feature value x is a
// float32, and for a float32 x  "(double)x <= threshold"  holds exactly when  x <= thr.
struct __align__(16) ForestNode {
    float thr;
    int left, right;
    int feat;
};
size_t forest_smem_bytes(int d);
// out_ids != null: node IDs relative to each tree's root (transform parity, int32 [n_q, ld_out]);
// else out_codes: 16-bit node codes [n_q, ld_out]
cudaError_t launch_forest_apply(const void *X, int x_dtype, long long ldx, long long n_q, int d,
                                const ForestNode *nodes, const int *roots, int n_trees,
                                uint16_t *out_codes, int *out_ids, long long ld_out, cudaStream_t st);

// ---- raster.cu (band-major raster blocks in, band-major result layers out) ------------------
constexpr int RASTER_GROUP = 1024;   // pixels per CTA of the mask / gather kernels
// pos [rows] <- valid flags, counts [groups + 1] <- exclusive group offsets (+ total), *total_out <- total
cudaError_t launch_raster_mask(const void *bands, int x_dtype, long long rows, int d, int use_nodata,
                               double nodata, int *pos, int *counts, int *total_out, cudaStream_t st);
// pos <- compacted row (or -1); xc [n_valid, d] <- the valid pixels' feature rows, pixel order kept
cudaError_t launch_raster_gather(const void *bands, int x_dtype, long long rows, int d, const int *offs,
                                 int *pos, void *xc, cudaStream_t st);
cudaError_t launch_raster_scatter_f64(const int *pos, long long rows, const double *src, int width,
                                      double fill, double *out, long long ld_out, cudaStream_t st);
cudaError_t launch_raster_scatter_i64(const int *pos, long long rows, const long long *src, int width,
                                      long long fill, long long *out, long long ld_out, cudaStream_t st);

// ---- misc ------------------------------------------------------------------------------
cudaError_t launch_fp32_peak(float *sink, int iters, int grid, cudaStream_t st);

}  // namespace sk

// Exact float64 epilogue of the search (SURVEY.md build-plan step 5):
//   refine_kernel  - re-evaluates the <= KC survivors of the FP32/TF32 search in float64,
//                    sorts them by (distance, index), proves with a rigorous error bound that
//                    no reference outside the survivor list can belong to the k nearest (the
//                    "certificate"), and finishes the row (self exclusion, sknnr's
//                    deterministic ordering, outputs, weighted average); refine2_kernel is the
//                    same for lists of <= 16 candidates with two queries per warp;
//   refine_lp_kernel - the same for Manhattan / Chebyshev indexes, one lane per candidate;
//   exact_kernel   - exhaustive float64 search for the rows whose certificate failed (and the
//                    engine for shapes the fast kernels do not cover); exact_hamming_kernel is the
//                    same for the weighted Hamming distance of node codes;
//   weighted_average_kernel - seam S3 with caller-supplied weights.
//
// The reference computes distances from the float64 expansion |x|^2 - 2x.y + |y|^2
// ($SP/sklearn/metrics/_pairwise_distances_reduction/_argkmin.pyx.tp:494-502) and returns
// sqrt of it (:285-295); here the k winners' distances come from direct float64 differences,
// which agree with it to the reference's own rounding noise (<= 1e-7 relative on raw features).
#include "common.cuh"
#include "kernels.h"

namespace sk {

constexpr int REFINE_WARPS = 8;

// Exact squared distance by direct float64 differences, summed in ONE fixed order shared by every
// kernel of this library (so all engines agree bit for bit): sixteen strided partial sums
//     p[h] = sum_j (zq[h + 16 j] - r[h + 16 j])^2,   j ascending,
// combined by the butterfly tree of a 16-lane shuffle reduction (xor 8, 4, 2, 1).
// dist2_lane is the partial of lane h of a half warp (coalesced: the half warp reads 128
// consecutive bytes of the reference row per load); dist2_serial replays the same tree in one
// thread.
__device__ __forceinline__ double dist2_lane(const double *__restrict__ zq, const double *__restrict__ r,
                                             int d, int h) {
    double acc = 0.0;
    for (int k = h; k < d; k += 16) {
        const double df = zq[k] - __ldg(r + k);
        acc = __fma_rn(df, df, acc);   // explicit: which product is fused must not be the compiler's choice
    }
    return acc;
}
// The same partial with the query's features already in registers (zr[j] = zq[h + 16 j], 0 past the
// end) and the loop unrolled: a missing feature contributes fma(0, 0, acc) = acc, so the bits equal
// dist2_lane's.
template <int DJ>
__device__ __forceinline__ double dist2_lane_regs(const double (&zr)[DJ], const double *__restrict__ r, int d,
                                                  int h) {
    double rv[DJ];
#pragma unroll
    for (int j = 0; j < DJ; ++j) rv[j] = (h + 16 * j < d) ? __ldg(r + h + 16 * j) : 0.0;
    double acc = 0.0;
#pragma unroll
    for (int j = 0; j < DJ; ++j) {
        const double df = zr[j] - rv[j];
        acc = __fma_rn(df, df, acc);
    }
    return acc;
}
__device__ __forceinline__ double dist2_reduce16(double acc) {
    acc += __shfl_xor_sync(SK_FULL, acc, 8);
    acc += __shfl_xor_sync(SK_FULL, acc, 4);
    acc += __shfl_xor_sync(SK_FULL, acc, 2);
    acc += __shfl_xor_sync(SK_FULL, acc, 1);
    return acc;
}
__device__ __forceinline__ double dist2_serial(const double *__restrict__ zq, const double *__restrict__ r,
                                               int d) {
    double p[16];
#pragma unroll
    for (int h = 0; h < 16; ++h) p[h] = 0.0;
    for (int k0 = 0; k0 < d; k0 += 16) {
#pragma unroll
        for (int h = 0; h < 16; ++h) {
            if (k0 + h < d) {
                const double df = zq[k0 + h] - r[k0 + h];
                p[h] = __fma_rn(df, df, p[h]);
            }
        }
    }
#pragma unroll
    for (int m = 8; m >= 1; m >>= 1) {
#pragma unroll
        for (int h = 0; h < m; ++h) p[h] = p[h] + p[h + m];   // == lane h after the xor-m shuffle step
    }
    return p[0];
}

// sqrt of the sorted squared distances: the padding lanes (+inf) take sqrt(1) instead, which keeps the
// warp on the square root's fast path; every other value, NaN included, goes through unchanged
__device__ __forceinline__ double sqrt_padded(double d2) {
    const bool pad = d2 == SK_INF_D;
    const double s = sqrt(pad ? 1.0 : d2);
    return pad ? SK_INF_D : s;
}

// Threshold (in the engine's scaled approximate-score units) for a second pass of the tensor engine over a
// row whose first-pass list was not certified.  `kth` is the exact k-th squared distance among the row's
// first-pass candidates, hence an upper bound of the true one: every reference that can still belong to the
// top k has approximate score <= (kth - |q|^2 + E) / thr_scale, E = eps_s (|q|^2 + max|r|^2).  A second pass
// that lists everything below a threshold a hair above that (rounded up to float) finds all of them, and
// its own certificate  kth' < thr * thr_scale + |q|^2 - E  then holds because kth' <= kth.
__device__ __forceinline__ float retry_threshold(double kth, double qn, const RefineArgs &a) {
    if (!(kth < SK_INF_D)) return SK_INF_F;   // fewer than k candidates so far (or NaN): start cold
    const double span = qn + a.r2max;
    double t = (kth - qn + a.eps_s * span) / a.thr_scale;
    t += 1e-6 * fabs(t) + 1e-9 * span / a.thr_scale;
    return __double2float_ru(t);
}

// DJ = ceil(d / 16) for d <= 64 (the query row lives in DJ registers per lane), 0 = any d
template <int DJ>
__global__ void __launch_bounds__(REFINE_WARPS * 32)
refine_kernel(RefineArgs a, FinishParams fp) {
    // (shuffle: the compiler then knows `warp` is warp-uniform and keeps what derives from it in uniform registers)
    const int warp = __shfl_sync(SK_FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const long long q = (long long)blockIdx.x * REFINE_WARPS + warp;
    if (q >= a.n_q || (a.n_rows_dev && q >= *a.n_rows_dev)) return;
    if (a.n_rows_dev && *a.n_rows_dev < a.bypass_rows) {   // the search was skipped: hand the row on
        if (lane == 0) a.fb_list[atomicAdd(a.fb_count, 1)] = a.row_map ? a.row_map[q] : (int)q;
        return;
    }
    const double *zq = a.z64 + q * a.d;

    // Exact squared distances of the candidates: each half warp takes one candidate per pass (its
    // 16 lanes read consecutive features, so a pass touches two lines of L2 instead of 32) and
    // reduces with a 16-lane butterfly; lane (i & 15) of the half warp keeps the result of pass i.
    const int half = lane >> 4, hl = lane & 15;
    const bool small = a.kc <= 16;      // lists of <= 16: candidate l ends up in lane l (16-lane sort)
    int id = 0x7fffffff;
    double d2 = SK_INF_D;
    const int my_c = lane < a.kc ? a.cand_idx[q * a.kc + lane] : -1;   // kc <= 32: one coalesced load
    double zr[DJ > 0 ? DJ : 1];
    if constexpr (DJ > 0) {
#pragma unroll
        for (int j = 0; j < DJ; ++j) zr[j] = (hl + 16 * j < a.d) ? zq[hl + 16 * j] : 0.0;
    }
#pragma unroll 4
    for (int i = 0; 2 * i < a.kc; ++i) {
        const int c = __shfl_sync(SK_FULL, my_c, (2 * i + half) & 31);
        const bool have = c >= 0 && c < a.n_ref;
        double acc = 0.0;
        if (have) {
            if constexpr (DJ > 0)
                acc = dist2_lane_regs<DJ>(zr, a.ref64 + (long long)c * a.d, a.d, hl);
            else
                acc = dist2_lane(zq, a.ref64 + (long long)c * a.d, a.d, hl);
        }
        acc = dist2_reduce16(acc);
        if (small) {
            const double other = __shfl_xor_sync(SK_FULL, acc, 16);   // the other half warp's candidate
            if ((lane >> 1) == i && lane < 16 && my_c >= 0 && my_c < a.n_ref) {
                id = my_c;
                d2 = (lane & 1) == half ? acc : other;
            }
        } else if (have && hl == (i & 15)) {
            id = c;
            d2 = acc;
        }
    }
    // |z_q - mu|^2 (lanes stride the features, then butterfly-reduce)
    double qn = 0.0;
    for (int k = lane; k < a.d; k += 32) {
        const double df = zq[k] - a.mu[k];
        qn += df * df;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) qn += __shfl_xor_sync(SK_FULL, qn, o);

    if (small)
        warp_sort_pairs<double, 16>(d2, id, lane);
    else
        warp_sort_pairs<double, 32>(d2, id, lane);

    const int kk = fp.k + (fp.exclude_self ? 1 : 0);
    const double kth = __shfl_sync(SK_FULL, d2, kk - 1);
    float thr = a.cand_thr[q * a.n_thr];
    for (int i = 1; i < a.n_thr; ++i) thr = fminf(thr, a.cand_thr[q * a.n_thr + i]);
    // every reference outside the list has approximate score >= thr, hence true squared
    // distance >= thr + |q|^2 - E with E = eps_s * (|q|^2 + max|r|^2)
    bool ok;
    if (thr == SK_INF_F) {
        ok = true;  // the list holds every reference
    } else {
        const double bound = (double)thr * a.thr_scale + qn - a.eps_s * (qn + a.r2max);
        ok = kth < bound && qn < a.qn_limit;
    }
    if (!ok) {
        if (lane == 0) {
            const int pos = atomicAdd(a.fb_count, 1);
            a.fb_list[pos] = a.row_map ? a.row_map[q] : (int)q;
            if (a.fb_thr) a.fb_thr[pos] = retry_threshold(kth, qn, a);
        }
        return;
    }
    finish_query(fp, q, sqrt_padded(d2), id, lane);
}

// Two queries per warp, one per 16-lane segment, for lists of <= 16 candidates and d <= 64 (the
// common case: the tensor and SIMT engines' k <= 14 lists): the sort network and everything in
// finish_query only ever needed 16 lanes, so this halves their instruction count per query.  A
// segment takes one candidate of ITS query per pass (16 lanes on 128 consecutive bytes of the
// reference row, 16-lane butterfly); lane i of the segment keeps candidate i.
template <int DJ>
__global__ void __launch_bounds__(REFINE_WARPS * 32)
refine2_kernel(RefineArgs a, FinishParams fp) {
    const int warp = __shfl_sync(SK_FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int seg = lane >> 4, hl = lane & 15;
    const long long n_rows = a.n_rows_dev ? min((long long)*a.n_rows_dev, a.n_q) : a.n_q;
    const long long q0 = ((long long)blockIdx.x * REFINE_WARPS + warp) * 2;
    if (q0 >= n_rows) return;                       // both segments idle: the whole warp leaves
    const bool live = q0 + seg < n_rows;            // odd tail: the second segment rides along
    const long long q = live ? q0 + seg : q0;
    if (a.n_rows_dev && n_rows < a.bypass_rows) {   // the search was skipped: hand the rows on
        if (live && hl == 0) a.fb_list[atomicAdd(a.fb_count, 1)] = a.row_map ? a.row_map[q] : (int)q;
        return;
    }
    const double *zq = a.z64 + q * a.d;
    double zr[DJ];
#pragma unroll
    for (int j = 0; j < DJ; ++j) zr[j] = (hl + 16 * j < a.d) ? zq[hl + 16 * j] : 0.0;
    const int my_c = hl < a.kc ? a.cand_idx[q * a.kc + hl] : -1;
    int id = 0x7fffffff;
    double d2 = SK_INF_D;
    auto take = [&](int i) {
        const int c = __shfl_sync(SK_FULL, my_c, i, 16);
        SK_CHECK(c >= -1 && c < a.n_ref);
        const bool have = c >= 0 && c < a.n_ref;
        double acc = 0.0;
        if (have) acc = dist2_lane_regs<DJ>(zr, a.ref64 + (long long)c * a.d, a.d, hl);
        acc = dist2_reduce16(acc);
        if (have && hl == i) {
            id = c;
            d2 = acc;
        }
    };
    // The tensor engine hands over two half lists of 8 slots, each filled from its first slot and
    // padded with -1 (typically 4 + 4 entries under the joint threshold): only the occupied prefix
    // of the two halves is visited, slot i and slot 8 + i per step.  Anything else: all slots.
    const unsigned vm = __ballot_sync(SK_FULL, my_c >= 0);
    int n_step = 8;
    if (a.kc == 16) {
        int worst = 0;
        bool prefix = true;
#pragma unroll
        for (int hlf = 0; hlf < 4; ++hlf) {
            const unsigned m = (vm >> (8 * hlf)) & 0xffu;
            const int n = __popc(m);
            prefix = prefix && (m == ((1u << n) - 1u));
            worst = max(worst, n);
        }
        if (prefix) n_step = worst;
        for (int i = 0; i < n_step; ++i) {
            take(i);
            take(8 + i);
        }
    } else {
#pragma unroll 4
        for (int i = 0; i < a.kc; ++i) take(i);
    }
    double qn = 0.0;
    for (int k = hl; k < a.d; k += 16) {
        const double df = zq[k] - a.mu[k];
        qn += df * df;
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) qn += __shfl_xor_sync(SK_FULL, qn, o);
    warp_sort_pairs<double, 16>(d2, id, hl);   // (segment lane: both segments sort ascending)

    const int kk = fp.k + (fp.exclude_self ? 1 : 0);
    const double kth = __shfl_sync(SK_FULL, d2, kk - 1, 16);
    float thr = a.cand_thr[q * a.n_thr];
    for (int i = 1; i < a.n_thr; ++i) thr = fminf(thr, a.cand_thr[q * a.n_thr + i]);
    bool ok = true;                                 // thr = +inf: the list holds every reference
    if (thr != SK_INF_F) ok = kth < (double)thr * a.thr_scale + qn - a.eps_s * (qn + a.r2max) && qn < a.qn_limit;
    if (live && !ok && hl == 0) {
        const int pos = atomicAdd(a.fb_count, 1);
        a.fb_list[pos] = a.row_map ? a.row_map[q] : (int)q;
        if (a.fb_thr) a.fb_thr[pos] = retry_threshold(kth, qn, a);
    }
    finish_query_w<16>(fp, q, sqrt_padded(d2), id, hl, live && ok);
}

cudaError_t launch_refine(const RefineArgs &a, const FinishParams &fp, cudaStream_t st) {
    if (a.n_q <= 0) return cudaSuccess;
    if (a.kc <= 16 && a.d <= 64) {
        const long long grid2 = (a.n_q + 2 * REFINE_WARPS - 1) / (2 * REFINE_WARPS);
        switch ((a.d + 15) / 16) {
            case 1: refine2_kernel<1><<<(unsigned)grid2, REFINE_WARPS * 32, 0, st>>>(a, fp); break;
            case 2: refine2_kernel<2><<<(unsigned)grid2, REFINE_WARPS * 32, 0, st>>>(a, fp); break;
            case 3: refine2_kernel<3><<<(unsigned)grid2, REFINE_WARPS * 32, 0, st>>>(a, fp); break;
            default: refine2_kernel<4><<<(unsigned)grid2, REFINE_WARPS * 32, 0, st>>>(a, fp); break;
        }
        return cudaGetLastError();
    }
    const long long grid = (a.n_q + REFINE_WARPS - 1) / REFINE_WARPS;
    switch (a.d <= 64 ? (a.d + 15) / 16 : 0) {
        case 1: refine_kernel<1><<<(unsigned)grid, REFINE_WARPS * 32, 0, st>>>(a, fp); break;
        case 2: refine_kernel<2><<<(unsigned)grid, REFINE_WARPS * 32, 0, st>>>(a, fp); break;
        case 3: refine_kernel<3><<<(unsigned)grid, REFINE_WARPS * 32, 0, st>>>(a, fp); break;
        case 4: refine_kernel<4><<<(unsigned)grid, REFINE_WARPS * 32, 0, st>>>(a, fp); break;
        default: refine_kernel<0><<<(unsigned)grid, REFINE_WARPS * 32, 0, st>>>(a, fp); break;
    }
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------
// Manhattan / Chebyshev: scikit-learn's ManhattanDistance64 / ChebyshevDistance64
// ($SP/sklearn/metrics/_dist_metrics.pyx.tp: d += fabs(x1[j] - x2[j]), resp. d = fmax(d, ...), j
// ascending, and the identity as rdist_to_dist), written with explicit roundings so that neither the
// order nor a contraction is the compiler's choice: the distances are bit-equal to the reference's.
template <int M>
__device__ __forceinline__ double dist_lp(const double *__restrict__ zq, const double *__restrict__ r, int d) {
    double acc = 0.0;
    for (int j = 0; j < d; ++j) {
        const double t = fabs(__dsub_rn(zq[j], __ldg(r + j)));
        acc = M == METRIC_L1 ? __dadd_rn(acc, t) : fmax(acc, t);
    }
    return acc;
}

// |q - mu| in the metric's norm, by the whole warp (lanes stride the features)
template <int M>
__device__ __forceinline__ double norm_lp_warp(const double *__restrict__ zq, const double *__restrict__ mu, int d,
                                               int lane) {
    double n = 0.0;
    for (int k = lane; k < d; k += 32) {
        const double t = fabs(zq[k] - mu[k]);
        n = M == METRIC_L1 ? n + t : fmax(n, t);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double other = __shfl_xor_sync(SK_FULL, n, o);
        n = M == METRIC_L1 ? n + other : fmax(n, other);
    }
    return n;
}

// One warp per query, one lane per candidate (kc <= 32): lane l recomputes candidate l's distance in
// scikit-learn's order, the warp sorts by (distance, index) and certifies the row when
//     kth < thr * thr_scale - eps_s * (|q - mu| + max_j |r_j - mu|)      (DESIGN.md §2, "Manhattan and Chebyshev")
// strictly, so that an exact tie with a reference outside the list goes to the exhaustive kernel.
// Every score is finite while |q - mu| < qn_limit (and the index's plots are below the same limit):
// thr = +inf then means that the list holds every reference.  A NaN norm never certifies.
template <int M, int SORT>
__global__ void __launch_bounds__(REFINE_WARPS * 32)
refine_lp_kernel(RefineArgs a, FinishParams fp) {
    const int warp = __shfl_sync(SK_FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const long long q = (long long)blockIdx.x * REFINE_WARPS + warp;
    if (q >= a.n_q) return;
    const double *zq = a.z64 + q * a.d;
    const int c = lane < a.kc ? a.cand_idx[q * a.kc + lane] : -1;
    SK_CHECK(c >= -1 && c < a.n_ref);
    int id = 0x7fffffff;
    double dist = SK_INF_D;
    if (c >= 0 && c < a.n_ref) {
        id = c;
        dist = dist_lp<M>(zq, a.ref64 + (long long)c * a.d, a.d);
    }
    const double qn = norm_lp_warp<M>(zq, a.mu, a.d, lane);
    warp_sort_pairs<double, SORT>(dist, id, lane);

    const int kk = fp.k + (fp.exclude_self ? 1 : 0);
    const double kth = __shfl_sync(SK_FULL, dist, kk - 1);
    const float thr = a.cand_thr[q];
    const bool ok = qn < a.qn_limit &&
                    (thr == SK_INF_F || kth < (double)thr * a.thr_scale - a.eps_s * (qn + a.r2max));
    if (!ok) {
        if (lane == 0) a.fb_list[atomicAdd(a.fb_count, 1)] = (int)q;
        return;
    }
    finish_query(fp, q, dist, id, lane);
}

cudaError_t launch_refine_lp(const RefineArgs &a, int metric, const FinishParams &fp, cudaStream_t st) {
    if (a.n_q <= 0) return cudaSuccess;
    if (a.kc > 32 || a.n_rows_dev || a.fb_thr || a.n_thr != 1) return cudaErrorInvalidValue;
    const long long grid = (a.n_q + REFINE_WARPS - 1) / REFINE_WARPS;
    // (lists of <= 16 sit in lanes 0..15: the sort network of 16 lanes suffices)
    if (metric == METRIC_L1 && a.kc <= 16)
        refine_lp_kernel<METRIC_L1, 16><<<(unsigned)grid, REFINE_WARPS * 32, 0, st>>>(a, fp);
    else if (metric == METRIC_L1)
        refine_lp_kernel<METRIC_L1, 32><<<(unsigned)grid, REFINE_WARPS * 32, 0, st>>>(a, fp);
    else if (metric == METRIC_LINF && a.kc <= 16)
        refine_lp_kernel<METRIC_LINF, 16><<<(unsigned)grid, REFINE_WARPS * 32, 0, st>>>(a, fp);
    else if (metric == METRIC_LINF)
        refine_lp_kernel<METRIC_LINF, 32><<<(unsigned)grid, REFINE_WARPS * 32, 0, st>>>(a, fp);
    else
        return cudaErrorInvalidValue;
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------
constexpr int EXACT_THREADS = 256;

// metric 0, 2 or 3
__device__ __forceinline__ double exact_pair(const ExactArgs &a, long long q, int j) {
    const double *zq = a.z64 + q * a.d;
    const double *r = a.ref64 + (long long)j * a.d;
    if (a.metric == 2) return dist_lp<METRIC_L1>(zq, r, a.d);
    if (a.metric == 3) return dist_lp<METRIC_LINF>(zq, r, a.d);
    return dist2_serial(zq, r, a.d);
}

// finish_query for k (+1) > 32, by the whole CTA: the kk selected neighbours arrive ascending by
// (distance, index) in sd / si (global scratch of the CTA, with room for the sort keys).  Same steps
// as finish_query_w: self exclusion, sknnr's ordering key, outputs, weighted average.  Large k is
// rare and rows reach this path one CTA at a time, so the sequential parts run on thread 0.
__device__ void finish_query_block(const FinishParams &p, long long q, double *sd, int *si, double *key,
                                   long long *sec, int kk) {
    __shared__ double sh_denom;
    __shared__ int sh_zero;
    const long long row = p.row_offset + q;
    if (threadIdx.x == 0) {
        if (p.exclude_self) {
            int pos = 0;
            for (int c = 0; c < kk; ++c)
                if ((long long)si[c] == row) { pos = c; break; }
            for (int c = pos; c + 1 < kk; ++c) {
                sd[c] = sd[c + 1];
                si[c] = si[c + 1];
            }
        }
        if (p.deterministic) {
            const double scale = fmax(sd[p.k - 1], 1.0);
            for (int c = 0; c < p.k; ++c) {
                key[c] = rint((sd[c] / scale) * p.round_scale) / p.round_scale;
                long long diff = (long long)si[c] - row;
                if (diff < 0) diff = -diff;
                sec[c] = (diff << 31) | (long long)si[c];
            }
            // the entries arrive sorted by distance and the key is monotone in it: an insertion sort
            // only ever moves entries inside a run of equal rounded keys
            for (int c = 1; c < p.k; ++c) {
                const double kc = key[c], dc = sd[c];
                const long long sc = sec[c];
                int j = c - 1;
                while (j >= 0 && (key[j] > kc || (key[j] == kc && sec[j] > sc))) {
                    key[j + 1] = key[j];
                    sec[j + 1] = sec[j];
                    sd[j + 1] = sd[j];
                    --j;
                }
                key[j + 1] = kc;
                sec[j + 1] = sc;
                sd[j + 1] = dc;
            }
            for (int c = 0; c < p.k; ++c) si[c] = (int)(sec[c] & 0x7fffffffLL);
        }
        int zero = 0;
        double denom = 0.0;
        if (p.weights == 2) {
            for (int c = 0; c < p.k; ++c) zero |= (sd[c] == 0.0);
            for (int c = 0; c < p.k; ++c) denom += zero ? (sd[c] == 0.0 ? 1.0 : 0.0) : 1.0 / sd[c];
        }
        sh_zero = zero;
        sh_denom = denom;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < p.k; c += blockDim.x) {
        if (p.out_dist) p.out_dist[q * p.k + c] = sd[c];
        if (p.out_idx) p.out_idx[q * p.k + c] = (long long)si[c];
    }
    if (p.weights != 0 && p.out_pred != nullptr) {
        for (int j = threadIdx.x; j < p.n_out; j += blockDim.x) {
            double num = 0.0;
            for (int c = 0; c < p.k; ++c) {
                const int ic = si[c];
                if (ic < 0 || ic >= p.n_ref) continue;
                const double yv = p.y[(long long)ic * p.n_out + j];
                if (p.weights == 1) {
                    num += yv;
                } else {
                    const double w = sh_zero ? (sd[c] == 0.0 ? 1.0 : 0.0) : 1.0 / sd[c];
                    num += yv * w;
                }
            }
            p.out_pred[q * p.n_out + j] = (p.weights == 1) ? (num / (double)p.k) : (num / sh_denom);
        }
    }
    __syncthreads();
}

// The exhaustive search of exact_kernel / exact_hamming_kernel; pair(q, j) is the float64 distance
template <class Pair>
__device__ __forceinline__ void exact_search(const ExactArgs &a, const FinishParams &fp, Pair pair) {
    __shared__ double red_d[EXACT_THREADS / 32];
    __shared__ int red_i[EXACT_THREADS / 32];
    __shared__ double sel_d_s[MAXK];
    __shared__ int sel_i_s[MAXK];
    // (shuffle: the compiler then knows `warp` is warp-uniform and keeps what derives from it in uniform registers)
    const int warp = __shfl_sync(SK_FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const long long n_rows = a.list ? (long long)(*a.count) : a.n_q;
    double *scr = a.scratch + (size_t)blockIdx.x * a.n_ref;
    const int kk = fp.k + (fp.exclude_self ? 1 : 0);
    // k (+1) > 32: the selection and the sort keys live in the CTA's slice of a.big
    //   [kk] distances | [kk] keys | [kk] secondary keys | [kk] indices
    const bool big = kk > MAXK;
    double *bigp = big ? a.big + (size_t)blockIdx.x * 4 * kk : nullptr;
    double *sel_d = big ? bigp : sel_d_s;
    int *sel_i = big ? reinterpret_cast<int *>(bigp + 3 * (size_t)kk) : sel_i_s;

    for (long long it = blockIdx.x; it < n_rows; it += gridDim.x) {
        const long long q = a.list ? (long long)a.list[it] : it;
        for (int j = threadIdx.x; j < a.n_ref; j += EXACT_THREADS) scr[j] = pair(q, j);
        __syncthreads();
        double last_d = -1.0;
        int last_i = -1;
        for (int r = 0; r < kk; ++r) {
            double bd = SK_INF_D;
            int bi = 0x7fffffff;
            for (int j = threadIdx.x; j < a.n_ref; j += EXACT_THREADS) {
                const double d = scr[j];
                const bool after = (d > last_d) || (d == last_d && j > last_i);
                if (after && pair_less<double>(d, j, bd, bi)) {
                    bd = d;
                    bi = j;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double od = __shfl_xor_sync(SK_FULL, bd, o);
                const int oi = __shfl_xor_sync(SK_FULL, bi, o);
                if (pair_less<double>(od, oi, bd, bi)) {
                    bd = od;
                    bi = oi;
                }
            }
            if (lane == 0) {
                red_d[warp] = bd;
                red_i[warp] = bi;
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                for (int w = 1; w < EXACT_THREADS / 32; ++w)
                    if (pair_less<double>(red_d[w], red_i[w], bd, bi)) {
                        bd = red_d[w];
                        bi = red_i[w];
                    }
                sel_d[r] = bd;
                sel_i[r] = bi;
                red_d[0] = bd;
                red_i[0] = bi;
            }
            __syncthreads();
            last_d = red_d[0];
            last_i = red_i[0];
            __syncthreads();
        }
        if (big) {
            if (a.metric == 0)
                for (int c = threadIdx.x; c < kk; c += EXACT_THREADS) sel_d[c] = sqrt(sel_d[c]);
            __syncthreads();
            finish_query_block(fp, q, sel_d, sel_i, bigp + kk, reinterpret_cast<long long *>(bigp + 2 * (size_t)kk), kk);
        } else if (warp == 0) {
            double d = (lane < kk) ? sel_d[lane] : SK_INF_D;
            const int id = (lane < kk) ? sel_i[lane] : 0x7fffffff;
            if (a.metric == 0) d = sqrt(d);
            finish_query(fp, q, d, id, lane);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(EXACT_THREADS)
exact_kernel(ExactArgs a, FinishParams fp) {
    exact_search(a, fp, [&](long long q, int j) { return exact_pair(a, q, j); });
}

// metric 1 (Code = uint16_t) or 4 (uint32_t): SciPy's weighted Hamming distance
template <class Code>
__global__ void __launch_bounds__(EXACT_THREADS)
exact_hamming_kernel(ExactArgs a, FinishParams fp) {
    exact_search(a, fp, [&](long long q, int j) {
        return hamming_numerator(static_cast<const Code *>(a.qcodes) + q * a.ldq,
                                 static_cast<const Code *>(a.rcodes) + (long long)j * a.n_trees, a.n_trees,
                                 a.w) / a.wsum;
    });
}

cudaError_t launch_exact(const ExactArgs &a, const FinishParams &fp, cudaStream_t st) {
    if (a.grid <= 0) return cudaSuccess;
    if (a.metric == 1)
        exact_hamming_kernel<uint16_t><<<a.grid, EXACT_THREADS, 0, st>>>(a, fp);
    else if (a.metric == 4)
        exact_hamming_kernel<uint32_t><<<a.grid, EXACT_THREADS, 0, st>>>(a, fp);
    else
        exact_kernel<<<a.grid, EXACT_THREADS, 0, st>>>(a, fp);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------
__global__ void weighted_average_kernel(const long long *__restrict__ idx,
                                        const double *__restrict__ w, long long n_q, int k,
                                        const double *__restrict__ y, int n_out,
                                        double *__restrict__ out) {
    // (shuffle: the compiler then knows `warp` is warp-uniform and keeps what derives from it in uniform registers)
    const int warp = __shfl_sync(SK_FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const long long q = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    if (q >= n_q) return;
    double denom = 0.0;
    for (int c = 0; c < k; ++c) denom += w[q * k + c];
    for (int j = lane; j < n_out; j += 32) {
        double num = 0.0;
        for (int c = 0; c < k; ++c) num += y[idx[q * k + c] * n_out + j] * w[q * k + c];
        out[q * n_out + j] = num / denom;
    }
}

__global__ void gather_rows_kernel(const double *__restrict__ z64, int d, const int *__restrict__ list,
                                   const int *__restrict__ count, double *__restrict__ z64c) {
    const long long n = *count;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n * d;
         e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / d;
        const int k = (int)(e - i * d);
        z64c[e] = z64[(long long)list[i] * d + k];
    }
}

cudaError_t launch_gather_rows(const double *z64, int d, const int *list, const int *count,
                               long long max_rows, double *z64c, cudaStream_t st) {
    if (max_rows <= 0) return cudaSuccess;
    const long long want = (max_rows * d + 255) / 256;
    const int grid = (int)(want < 1184 ? want : 1184);
    gather_rows_kernel<<<grid, 256, 0, st>>>(z64, d, list, count, z64c);
    return cudaGetLastError();
}

cudaError_t launch_weighted_average(const long long *idx, const double *w, long long n_q, int k,
                                    const double *y, int n_out, double *out_pred,
                                    cudaStream_t st) {
    if (n_q <= 0) return cudaSuccess;
    const int warps = 8;
    const long long grid = (n_q + warps - 1) / warps;
    weighted_average_kernel<<<(unsigned)grid, warps * 32, 0, st>>>(idx, w, n_q, k, y, n_out,
                                                                  out_pred);
    return cudaGetLastError();
}

}  // namespace sk

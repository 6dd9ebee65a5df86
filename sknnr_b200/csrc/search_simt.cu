// Fused FP32 distance + top-KC candidate selection (north_star pieces 2 + 3), SIMT engine.
//
// Replaces the hot loop of scikit-learn's EuclideanArgKmin64
// ($SP/sklearn/metrics/_pairwise_distances_reduction/_argkmin.pyx.tp:401-510: dgemm tile,
// d2 = |x|^2 - 2x.y + |y|^2, one heap test per pair), reached from
// ref:src/sknnr/_base.py:162-164.  The n_q x n_ref distance matrix never reaches HBM.
//
// Work decomposition (one CTA = 384 queries, 12 warps; lane 0 of warp 0 doubles as the TMA
// producer, so the warp count stays a multiple of 4 and the register budget is 168/thread):
//   * the CTA's query tile image [dpad][384] f32 (pre-scaled by -2, centroid-shifted) is
//     staged once with one 1-D TMA bulk copy;
//   * reference tiles of 64 plots, image [(dpad+1)][64] f32 whose last row holds |r|^2, stream
//     through an NSTAGE-deep ring filled with cp.async.bulk + mbarrier complete_tx and
//     released by the compute warps through "empty" mbarriers;
//   * each compute warp owns 32 queries; lanes form a 4 (query groups) x 8 (reference groups)
//     grid and every thread keeps an 8 query x 8 reference register tile of FP32 scores
//     s = |r|^2 - 2 q.r accumulated with packed FFMA2 (two references per instruction);
//   * selection: one compare per pair against the query's current KC-th best score; hits
//     (k*ln(n_ref/k) per query) are inserted into the query's sorted list, which the 8 lanes
//     sharing the query keep in registers (width-8 shuffles; the four lane groups of a warp
//     insert into four queries at once).  No atomics, no barrier, no shared memory (lists of
//     more than 16 entries fall back to a shared-memory list owned by the warp).
//
// Output: for every query the KC best references by approximate score (ascending) and the
// KC-th score.  Exact float64 distances, ordering and the certificate that no better
// reference was missed are the refine kernel's job (refine.cu).
#include "common.cuh"
#include "kernels.h"

namespace sk {

// M = METRIC_L2: Euclidean scores as above.  M = METRIC_L1 / METRIC_LINF (Manhattan / Chebyshev): both
// images hold -2 (x - mu), the bias row holds 0 (+inf for padding plots), and a score is the FP32
// sum (max) of |q_k - r_k| over the features, twice the approximate L1 (L-inf) distance.
template <int KC, int M>
__global__ void __launch_bounds__(SEARCH_THREADS, 1)
search_simt_kernel(const float *__restrict__ qimg, const float *__restrict__ rimg, int dpad,
                   int n_rtiles, int nstage, long long n_q, int *__restrict__ cand_idx,
                   float *__restrict__ cand_thr, const int *__restrict__ n_rows_dev, int spread_ctas,
                   int bypass_rows) {
    long long qtile = blockIdx.x;
    int wpc = NCOMPUTE_WARPS, woff = 0;   // warps of this CTA that have rows, first warp slot of the tile it serves
    if (n_rows_dev) {
        // Compacted launch (second stage of the cascade): the row count is only known on the device and is
        // usually a fraction of a percent of the chunk.  One CTA per 384 rows would leave most SMs idle for
        // a full scan of the reference set, so the rows are dealt out in units of one warp (32 rows) over
        // up to spread_ctas CTAs: CTA b serves wpc consecutive warp slots of a query tile, wpc the smallest
        // divisor of 12 that covers the rows, and its other warps retire at once.
        const long long n_dev = *n_rows_dev;
        if (n_dev < bypass_rows) return;   // too few rows to be worth a scan: they go to the exhaustive kernel
        n_q = min(n_q, n_dev);
        const long long n_w = (n_q + 31) / 32;
        const long long per = spread_ctas > 0 ? (n_w + spread_ctas - 1) / spread_ctas : NCOMPUTE_WARPS;
        wpc = per <= 1 ? 1 : per <= 2 ? 2 : per <= 3 ? 3 : per <= 4 ? 4 : per <= 6 ? 6 : NCOMPUTE_WARPS;
        const long long w0 = (long long)blockIdx.x * wpc;
        if (w0 >= n_w) return;
        qtile = w0 / NCOMPUTE_WARPS;
        woff = (int)(w0 - qtile * NCOMPUTE_WARPS);
    }
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int rtile_floats = (dpad + 1) * RTILE;
    float *Qs = reinterpret_cast<float *>(smem_raw);
    float *Rs = Qs + (size_t)dpad * QTILE;
    constexpr bool kRegLists = KC <= 16;          // lists live in registers (8-lane groups)
    constexpr int EPL = kRegLists ? KC / 8 : 1;   // list entries per lane
    constexpr int kListSlots = kRegLists ? 0 : QTILE * KC;
    float *list_s = Rs + (size_t)nstage * rtile_floats;
    int *list_i = reinterpret_cast<int *>(list_s + kListSlots);
    uint64_t *full = reinterpret_cast<uint64_t *>(list_i + kListSlots);
    uint64_t *empty = full + nstage;
    uint64_t *qbar = empty + nstage;

    // (shuffle: the compiler then knows `warp` is warp-uniform and keeps what derives from it in uniform registers)
    const int warp0 = __shfl_sync(SK_FULL, (int)(threadIdx.x >> 5), 0);
    const int warp = warp0 + woff;   // warp slot of the query tile
    const int lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < nstage; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], wpc);
        }
        mbar_init(qbar, 1);
        fence_mbar_init();
    }
    for (int e = threadIdx.x; e < kListSlots; e += SEARCH_THREADS) {
        list_s[e] = SK_INF_F;
        list_i[e] = -1;
    }
    __syncthreads();
    if (warp0 >= wpc) return;

    // ---------------- TMA producer: lane 0 of warp 0, inline ----------------
    // Tile t+nstage-2 is requested at the top of iteration t, so the slot it overwrites was
    // released two iterations ago and the wait below is normally already satisfied.
    const uint32_t rbytes = (uint32_t)rtile_floats * 4u;
    auto issue_tile = [&](int tn) {
        const int sn = tn % nstage;
        if (tn >= nstage) mbar_wait(&empty[sn], ((tn / nstage) - 1) & 1);
        mbar_expect_tx(&full[sn], rbytes);
        bulk_g2s(Rs + (size_t)sn * rtile_floats, rimg + (size_t)tn * rtile_floats, rbytes, &full[sn]);
    };
    if (threadIdx.x == 0) {
        const uint32_t qbytes = (uint32_t)dpad * QTILE * 4u;
        mbar_expect_tx(qbar, qbytes);
        bulk_g2s(Qs, qimg + (size_t)qtile * dpad * QTILE, qbytes, qbar);
        for (int tn = 0; tn < nstage - 1 && tn < n_rtiles; ++tn) issue_tile(tn);
    }

    // ---------------- compute warps ----------------
    const int ty = lane >> 3;  // query group 0..3
    const int tx = lane & 7;   // reference group 0..7
    const float *qp = Qs + warp * 32 + ty * 4;
    float thr[8];
    float lk[8][EPL];  // register lists: lane tx holds positions tx*EPL.. of its 8 queries
    int li[8][EPL];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        thr[i] = SK_INF_F;
#pragma unroll
        for (int e = 0; e < EPL; ++e) {
            lk[i][e] = SK_INF_F;
            li[i][e] = -1;
        }
    }

    mbar_wait(qbar, 0);

    for (int t = 0; t < n_rtiles; ++t) {
        if (threadIdx.x == 0 && t >= 1 && t + nstage - 2 < n_rtiles) issue_tile(t + nstage - 2);
        __syncwarp();
        const int s = t % nstage;
        mbar_wait(&full[s], (t / nstage) & 1);
        const float *rp = Rs + (size_t)s * rtile_floats + tx * 4;

        float2 acc[8][4];
        {
            const float4 n0 = *reinterpret_cast<const float4 *>(rp + dpad * RTILE);
            const float4 n1 = *reinterpret_cast<const float4 *>(rp + dpad * RTILE + 32);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                acc[i][0] = make_float2(n0.x, n0.y);
                acc[i][1] = make_float2(n0.z, n0.w);
                acc[i][2] = make_float2(n1.x, n1.y);
                acc[i][3] = make_float2(n1.z, n1.w);
            }
        }
        if constexpr (M == METRIC_L2) {
            for (int k0 = 0; k0 < dpad; k0 += 8) {
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {
                    const int k = k0 + kk;
                    const float4 qa = *reinterpret_cast<const float4 *>(qp + k * QTILE);
                    const float4 qb = *reinterpret_cast<const float4 *>(qp + k * QTILE + 16);
                    const float4 ra = *reinterpret_cast<const float4 *>(rp + k * RTILE);
                    const float4 rb = *reinterpret_cast<const float4 *>(rp + k * RTILE + 32);
                    const float2 r0 = make_float2(ra.x, ra.y), r1 = make_float2(ra.z, ra.w);
                    const float2 r2 = make_float2(rb.x, rb.y), r3 = make_float2(rb.z, rb.w);
                    const float qv[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float2 qd = make_float2(qv[i], qv[i]);
                        acc[i][0] = __ffma2_rn(qd, r0, acc[i][0]);
                        acc[i][1] = __ffma2_rn(qd, r1, acc[i][1]);
                        acc[i][2] = __ffma2_rn(qd, r2, acc[i][2]);
                        acc[i][3] = __ffma2_rn(qd, r3, acc[i][3]);
                    }
                }
            }
        } else {
            // one FADD2 forms the differences q_k - r_k of two references; L1 adds their magnitudes
            // with a second FADD2 (|.| is an operand modifier), L-inf takes two FMNMX
            for (int k0 = 0; k0 < dpad; k0 += 8) {
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {
                    const int k = k0 + kk;
                    const float4 qa = *reinterpret_cast<const float4 *>(qp + k * QTILE);
                    const float4 qb = *reinterpret_cast<const float4 *>(qp + k * QTILE + 16);
                    const float4 ra = *reinterpret_cast<const float4 *>(rp + k * RTILE);
                    const float4 rb = *reinterpret_cast<const float4 *>(rp + k * RTILE + 32);
                    const float2 nr[4] = {make_float2(-ra.x, -ra.y), make_float2(-ra.z, -ra.w),
                                          make_float2(-rb.x, -rb.y), make_float2(-rb.z, -rb.w)};
                    const float qv[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float2 qd = make_float2(qv[i], qv[i]);
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const float2 t = __fadd2_rn(qd, nr[c]);
                            if constexpr (M == METRIC_L1) {
                                acc[i][c] = __fadd2_rn(acc[i][c], make_float2(fabsf(t.x), fabsf(t.y)));
                            } else {
                                acc[i][c].x = fmaxf(acc[i][c].x, fabsf(t.x));
                                acc[i][c].y = fmaxf(acc[i][c].y, fabsf(t.y));
                            }
                        }
                    }
                }
            }
        }
        // the staged tile is no longer needed: hand the slot back to the producer
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);

        // ---------------- selection ----------------
        bool rowhit[8];
        bool anyhit = false;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float m0 = fminf(fminf(acc[i][0].x, acc[i][0].y), fminf(acc[i][1].x, acc[i][1].y));
            const float m1 = fminf(fminf(acc[i][2].x, acc[i][2].y), fminf(acc[i][3].x, acc[i][3].y));
            rowhit[i] = fminf(m0, m1) < thr[i];
            anyhit |= rowhit[i];
        }
        if (__any_sync(SK_FULL, anyhit)) {
            const int idbase = t * RTILE;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const unsigned mrow = __ballot_sync(SK_FULL, rowhit[i]);
                if (mrow == 0) continue;
                if constexpr (kRegLists) {
                    const float sc[8] = {acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y,
                                         acc[i][2].x, acc[i][2].y, acc[i][3].x, acc[i][3].y};
                    unsigned hm = 0;
#pragma unroll
                    for (int c = 0; c < 8; ++c) hm |= (sc[c] < thr[i]) ? (1u << c) : 0u;
                    drain_row<EPL, float, false>(sc, hm, lk[i], li[i], thr[i], idbase, 0x7fffffff,
                                                 tx, ty);
                } else {
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const float sc = (c & 1) ? acc[i][c >> 1].y : acc[i][c >> 1].x;
                        unsigned m = __ballot_sync(SK_FULL, sc < thr[i]);
                        while (m) {
                            const int src = __ffs(m) - 1;
                            m &= m - 1;
                            const float s_l = __shfl_sync(SK_FULL, sc, src);
                            const int ty_l = src >> 3, tx_l = src & 7;
                            const int qs = tile_query_slot(warp, ty_l, i);
                            const int id_l = idbase + tile_ref_slot(tx_l, c);
                            float nthr;
                            int nid;
                            list_insert<KC, float, false>(list_s, list_i, qs, s_l, id_l, lane, nthr, nid);
                            if (ty == ty_l) thr[i] = nthr;
                        }
                    }
                }
            }
        }
    }

    // ---------------- write candidates ----------------
    if constexpr (kRegLists) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const long long q = qtile * QTILE + tile_query_slot(warp, ty, i);
            if (q < n_q) {
#pragma unroll
                for (int e = 0; e < EPL; ++e) cand_idx[q * KC + tx * EPL + e] = li[i][e];
                if (tx == 7) cand_thr[q] = lk[i][EPL - 1];
            }
        }
    } else {
        for (int ql = 0; ql < 32; ++ql) {
            const int qs = warp * 32 + ql;
            const long long q = qtile * QTILE + qs;
            if (q >= n_q) break;
            if (lane < KC) {
                cand_idx[q * KC + lane] = list_i[qs * KC + lane];
                if (lane == KC - 1) cand_thr[q] = list_s[qs * KC + lane];
            }
        }
    }
}

size_t search_simt_smem_bytes(int dpad, int kc, int nstage) {
    const size_t lists = kc <= 16 ? 0 : (size_t)QTILE * kc * 8;  // <= 16: register lists
    return (size_t)dpad * QTILE * 4 + (size_t)nstage * (dpad + 1) * RTILE * 4 + lists +
           (size_t)(2 * nstage + 1) * 8;
}

int search_simt_pick_stages(int dpad, int kc) {
    for (int s = 4; s >= 2; --s)
        if (search_simt_smem_bytes(dpad, kc, s) <= 227 * 1024) return s;
    return 0;
}

template <int KC, int M>
static cudaError_t launch_kc(const float *qimg, const float *rimg, int dpad, int n_rtiles,
                             long long n_q, int *cand_idx, float *cand_thr, const int *n_rows_dev,
                             int spread_ctas, int bypass_rows, cudaStream_t st) {
    const int nstage = search_simt_pick_stages(dpad, KC);
    if (nstage == 0) return cudaErrorInvalidValue;
    const size_t smem = search_simt_smem_bytes(dpad, KC, nstage);
    cudaError_t e = cudaFuncSetAttribute(search_simt_kernel<KC, M>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    const long long n_qtiles = (n_q + QTILE - 1) / QTILE;
    const long long grid = n_rows_dev && spread_ctas > n_qtiles ? spread_ctas : n_qtiles;
    search_simt_kernel<KC, M><<<(unsigned)grid, SEARCH_THREADS, smem, st>>>(
        qimg, rimg, dpad, n_rtiles, nstage, n_q, cand_idx, cand_thr, n_rows_dev, spread_ctas, bypass_rows);
    return cudaGetLastError();
}

template <int M>
static cudaError_t launch_metric(const float *qimg, const float *rimg, int dpad, int n_rtiles, long long n_q,
                                 int kc, int *cand_idx, float *cand_thr, const int *n_rows_dev, int spread_ctas,
                                 int bypass_rows, cudaStream_t st) {
    switch (kc) {
        case 8: return launch_kc<8, M>(qimg, rimg, dpad, n_rtiles, n_q, cand_idx, cand_thr, n_rows_dev, spread_ctas, bypass_rows, st);
        case 16: return launch_kc<16, M>(qimg, rimg, dpad, n_rtiles, n_q, cand_idx, cand_thr, n_rows_dev, spread_ctas, bypass_rows, st);
        case 32: return launch_kc<32, M>(qimg, rimg, dpad, n_rtiles, n_q, cand_idx, cand_thr, n_rows_dev, spread_ctas, bypass_rows, st);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_search_simt(const float *qimg, const float *rimg, int dpad, int n_rtiles,
                               long long n_q, int kc, int *cand_idx, float *cand_thr,
                               const int *n_rows_dev, int spread_ctas, int bypass_rows, cudaStream_t st,
                               int metric) {
    if (n_q <= 0) return cudaSuccess;
    switch (metric) {
        case METRIC_L2: return launch_metric<METRIC_L2>(qimg, rimg, dpad, n_rtiles, n_q, kc, cand_idx, cand_thr, n_rows_dev, spread_ctas, bypass_rows, st);
        case METRIC_L1: return launch_metric<METRIC_L1>(qimg, rimg, dpad, n_rtiles, n_q, kc, cand_idx, cand_thr, n_rows_dev, spread_ctas, bypass_rows, st);
        case METRIC_LINF: return launch_metric<METRIC_LINF>(qimg, rimg, dpad, n_rtiles, n_q, kc, cand_idx, cand_thr, n_rows_dev, spread_ctas, bypass_rows, st);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace sk

// Integer Hamming distance over random-forest terminal-node IDs + fused top-k
// (north_star piece 4).  Replaces sklearn's brute Hamming branch -> scipy cdist_hamming
// ($SP/sklearn/neighbors/_base.py:879-908,715-754; $SP/scipy/spatial/distance.py:1718-1723)
// reached by RFNNRegressor with metric="hamming" (ref:src/sknnr/_weighted_trees.py:46-59).
//
// With equal tree weights (RFNN: ref:src/sknnr/transformers/_rfnode_transformer.py:227-232,
// ref:src/sknnr/_weighted_trees.py:74-75) the float64 distance is a strictly increasing
// function of the integer mismatch count, so the kernel ranks by (count, index) - bit-exact -
// and a host-built table turns counts into the float64 values SciPy produces.
//
// Node IDs only need equality, so the host maps them to dense 16-bit codes < 31744.  Read as
// IEEE half precision those codes are distinct non-negative finite numbers, hence two trees are
// compared per instruction with HSET2.NE (1.0 / 0.0 per half) and accumulated with HADD2
// (exact up to 2048 per half): one instruction per ID compare.
//
// Unequal tree weights (GBNNRegressor's train-improvement weights, ref:src/sknnr/transformers/
// _gbnode_transformer.py:20-56,288-310; RFNN with user forest_weights) make the distance a
// float64 sum whose order is no longer that of the count.  The same kernel then runs as a FILTER
// on 16-bit fixed-point weights: HSET2.BM.NE turns two trees into 0xffff/0 half masks, one PRMT
// gathers four trees' mask bytes (-1 / 0 as s8) and two IDP.2A add  -w_t  per mismatching tree
// into one s32 accumulator - 1.25 instructions per ID compare, exact integer sums, no ordering
// effects.  hamming_refine_kernel recomputes the float64 distances of the surviving candidates
// in SciPy's summation order and certifies the top k against the quantisation error bound;
// uncertified rows go to the exhaustive float64 kernel (refine.cu).
//
// Same decomposition as search_simt.cu (384 queries per CTA, 12 warps, lane 0 of warp 0 issues
// the TMA copies, 8x8 register tile of accumulators per thread), except that the tree axis is long
// (T = 500), so both operands stream through the shared-memory ring in chunks of 64 trees:
// stage = query chunk [32 words][384] + reference chunk [32 words][64] (56 KB).
#include "common.cuh"
#include "kernels.h"

namespace sk {

constexpr int HAM_QCH = HAM_WC * QTILE;   // u32 words of a query chunk
constexpr int HAM_RCH = HAM_WC * RTILE;   // u32 words of a reference chunk
constexpr int HAM_STAGE = HAM_QCH + HAM_RCH;

// ---- pack: u16 codes [n, ldc] -> [n_tiles][n_chunks][HAM_WC][tile] u32 -----------------
__global__ void __launch_bounds__(256)
hamming_pack_kernel(const uint16_t *__restrict__ codes, long long n, long long ldc, int n_trees,
                    int n_chunks, int tile, uint16_t pad_code, uint32_t *__restrict__ img) {
    constexpr int SUB = 128;  // rows transposed per pass through shared memory
    __shared__ uint32_t buf[HAM_WC][SUB + 1];
    const long long tileno = blockIdx.x;
    const int chunk = blockIdx.y;
    uint32_t *out = img + ((size_t)tileno * n_chunks + chunk) * HAM_WC * tile;
    for (int sub = 0; sub < tile; sub += SUB) {
        const int nsub = min(SUB, tile - sub);
        const long long row0 = tileno * tile + sub;
        for (int e = threadIdx.x; e < nsub * HAM_WC; e += 256) {
            const int r = e / HAM_WC, w = e - r * HAM_WC;
            const long long row = row0 + r;
            const int t0 = 2 * (chunk * HAM_WC + w);
            uint32_t lo = 0, hi = 0;
            if (row < n) {
                if (t0 < n_trees) lo = codes[row * ldc + t0];
                if (t0 + 1 < n_trees) hi = codes[row * ldc + t0 + 1];
            } else {
                if (t0 < n_trees) lo = pad_code;
                if (t0 + 1 < n_trees) hi = pad_code;
            }
            buf[w][r] = lo | (hi << 16);
        }
        __syncthreads();
        for (int e = threadIdx.x; e < nsub * HAM_WC; e += 256) {
            const int w = e / nsub, r = e - w * nsub;
            out[(size_t)w * tile + sub + r] = buf[w][r];
        }
        __syncthreads();
    }
}

cudaError_t launch_hamming_pack(const uint16_t *codes, long long n, long long ldc, int n_trees,
                                int n_chunks, int tile, uint16_t pad_code, uint32_t *img,
                                cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const long long tiles = (n + tile - 1) / tile;
    dim3 grid((unsigned)tiles, (unsigned)n_chunks);
    hamming_pack_kernel<<<grid, 256, 0, st>>>(codes, n, ldc, n_trees, n_chunks, tile, pad_code, img);
    return cudaGetLastError();
}

// ---- search ---------------------------------------------------------------------------
__device__ __forceinline__ int dp2a_lo_u16_s8(uint32_t a, uint32_t b, int c) {
    int d;
    asm("dp2a.lo.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int dp2a_hi_u16_s8(uint32_t a, uint32_t b, int c) {
    int d;
    asm("dp2a.hi.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// WTD = false: mismatch counts (equal weights).  WTD = true: sums of the 16-bit fixed-point
// weights wq [n_chunks * HAM_WC] (two trees per word, like the code images) of the mismatching trees.
template <int KC, bool WTD>
__global__ void __launch_bounds__(SEARCH_THREADS, 1)
hamming_search_kernel(const uint32_t *__restrict__ qimg, const uint32_t *__restrict__ rimg,
                      const uint32_t *__restrict__ wq, int n_chunks, int n_rtiles, int nstage,
                      long long n_q, int n_ref, int *__restrict__ cand_idx,
                      int *__restrict__ cand_cnt) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint32_t *stage0 = reinterpret_cast<uint32_t *>(smem_raw);
    constexpr bool kRegLists = KC <= 16;          // lists live in registers (8-lane groups)
    constexpr int EPL = kRegLists ? KC / 8 : 1;
    constexpr int kListSlots = kRegLists ? 0 : QTILE * KC;
    int *list_c = reinterpret_cast<int *>(stage0 + (size_t)nstage * HAM_STAGE);
    int *list_i = list_c + kListSlots;
    uint64_t *full = reinterpret_cast<uint64_t *>(list_i + kListSlots);
    uint64_t *empty = full + nstage;
    uint32_t *wq_s = reinterpret_cast<uint32_t *>(empty + nstage);   // WTD only

    // (shuffle: the compiler then knows `warp` is warp-uniform and keeps what derives from it in uniform registers)
    const int warp = __shfl_sync(SK_FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < nstage; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], NCOMPUTE_WARPS);
        }
        fence_mbar_init();
    }
    if constexpr (WTD)
        for (int e = threadIdx.x; e < n_chunks * HAM_WC; e += SEARCH_THREADS) wq_s[e] = wq[e];
    for (int e = threadIdx.x; e < kListSlots; e += SEARCH_THREADS) {
        list_c[e] = 0x7fffffff;
        list_i[e] = 0x7fffffff;
    }
    __syncthreads();

    const long long qtile = blockIdx.x;
    const int n_steps = n_rtiles * n_chunks;

    // TMA producer: lane 0 of warp 0, inline (step+nstage-2 is requested at the top of `step`)
    auto issue_step = [&](int sn_step) {
        const int sn = sn_step % nstage;
        const int tt = sn_step / n_chunks, cc = sn_step - tt * n_chunks;
        if (sn_step >= nstage) mbar_wait(&empty[sn], ((sn_step / nstage) - 1) & 1);
        uint32_t *dst = stage0 + (size_t)sn * HAM_STAGE;
        mbar_expect_tx(&full[sn], HAM_STAGE * 4u);
        bulk_g2s(dst, qimg + ((size_t)qtile * n_chunks + cc) * HAM_QCH, HAM_QCH * 4u, &full[sn]);
        bulk_g2s(dst + HAM_QCH, rimg + ((size_t)tt * n_chunks + cc) * HAM_RCH, HAM_RCH * 4u, &full[sn]);
    };
    if (threadIdx.x == 0)
        for (int sn_step = 0; sn_step < nstage - 1 && sn_step < n_steps; ++sn_step) issue_step(sn_step);

    const int ty = lane >> 3, tx = lane & 7;
    int thr[8];
    int lk[8][EPL], li[8][EPL];  // register lists (counts, ids)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        thr[i] = 0x7fffffff;
#pragma unroll
        for (int e = 0; e < EPL; ++e) {
            lk[i][e] = 0x7fffffff;
            li[i][e] = 0x7fffffff;
        }
    }

    __half2 acc[8][8];
    int wacc[8][8];   // WTD: minus the fixed-point weight sums
    int step = 0;
    for (int t = 0; t < n_rtiles; ++t) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                acc[i][j] = __floats2half2_rn(0.f, 0.f);
                wacc[i][j] = 0;
            }

        for (int c = 0; c < n_chunks; ++c, ++step) {
            if (threadIdx.x == 0 && step >= 1 && step + nstage - 2 < n_steps) issue_step(step + nstage - 2);
            __syncwarp();
            const int s = step % nstage;
            mbar_wait(&full[s], (step / nstage) & 1);
            const uint32_t *qp = stage0 + (size_t)s * HAM_STAGE + warp * 32 + ty * 4;
            const uint32_t *rp = stage0 + (size_t)s * HAM_STAGE + HAM_QCH + tx * 4;
            if constexpr (WTD) {
                const uint32_t *wp = wq_s + c * HAM_WC;
#pragma unroll 2
                for (int w = 0; w < HAM_WC; w += 2) {
                    uint32_t qv[2][8], rv[2][8];
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const uint4 qa = *reinterpret_cast<const uint4 *>(qp + (w + h) * QTILE);
                        const uint4 qb = *reinterpret_cast<const uint4 *>(qp + (w + h) * QTILE + 16);
                        const uint4 ra = *reinterpret_cast<const uint4 *>(rp + (w + h) * RTILE);
                        const uint4 rb = *reinterpret_cast<const uint4 *>(rp + (w + h) * RTILE + 32);
                        qv[h][0] = qa.x; qv[h][1] = qa.y; qv[h][2] = qa.z; qv[h][3] = qa.w;
                        qv[h][4] = qb.x; qv[h][5] = qb.y; qv[h][6] = qb.z; qv[h][7] = qb.w;
                        rv[h][0] = ra.x; rv[h][1] = ra.y; rv[h][2] = ra.z; rv[h][3] = ra.w;
                        rv[h][4] = rb.x; rv[h][5] = rb.y; rv[h][6] = rb.z; rv[h][7] = rb.w;
                    }
                    const uint32_t w01 = wp[w], w23 = wp[w + 1];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const __half2 q0 = *reinterpret_cast<const __half2 *>(&qv[0][i]);
                        const __half2 q1 = *reinterpret_cast<const __half2 *>(&qv[1][i]);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const uint32_t m0 = __hne2_mask(q0, *reinterpret_cast<const __half2 *>(&rv[0][j]));
                            const uint32_t m1 = __hne2_mask(q1, *reinterpret_cast<const __half2 *>(&rv[1][j]));
                            const uint32_t m4 = __byte_perm(m0, m1, 0x6420);   // one -1/0 byte per tree
                            wacc[i][j] = dp2a_lo_u16_s8(w01, m4, wacc[i][j]);
                            wacc[i][j] = dp2a_hi_u16_s8(w23, m4, wacc[i][j]);
                        }
                    }
                }
            } else {
#pragma unroll 4
            for (int w = 0; w < HAM_WC; ++w) {
                const uint4 qa = *reinterpret_cast<const uint4 *>(qp + w * QTILE);
                const uint4 qb = *reinterpret_cast<const uint4 *>(qp + w * QTILE + 16);
                const uint4 ra = *reinterpret_cast<const uint4 *>(rp + w * RTILE);
                const uint4 rb = *reinterpret_cast<const uint4 *>(rp + w * RTILE + 32);
                const uint32_t qv[8] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
                const uint32_t rv[8] = {ra.x, ra.y, ra.z, ra.w, rb.x, rb.y, rb.z, rb.w};
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const __half2 qh = *reinterpret_cast<const __half2 *>(&qv[i]);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const __half2 rh = *reinterpret_cast<const __half2 *>(&rv[j]);
                        acc[i][j] = __hadd2(acc[i][j], __hne2(qh, rh));
                    }
                }
            }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
        }

        // ---- selection on exact integer counts, ties broken by the lowest index ----
        int cnt[8][8];
        bool rowhit[8];
        bool anyhit = false;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int mn = 0x7fffffff;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if constexpr (WTD)
                    cnt[i][j] = -wacc[i][j];
                else
                    cnt[i][j] = (int)(__low2float(acc[i][j]) + __high2float(acc[i][j]));
                mn = min(mn, cnt[i][j]);
            }
            rowhit[i] = mn <= thr[i];
            anyhit |= rowhit[i];
        }
        if (__any_sync(SK_FULL, anyhit)) {
            const int idbase = t * RTILE;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const unsigned mrow = __ballot_sync(SK_FULL, rowhit[i]);
                if (mrow == 0) continue;
                if constexpr (kRegLists) {
                    unsigned hm = 0;
#pragma unroll
                    for (int c = 0; c < 8; ++c) hm |= (cnt[i][c] <= thr[i]) ? (1u << c) : 0u;
                    drain_row<EPL, int, true>(cnt[i], hm, lk[i], li[i], thr[i], idbase, n_ref, tx, ty);
                } else {
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const int myid = idbase + tile_ref_slot(tx, c);
                        unsigned m = __ballot_sync(SK_FULL, cnt[i][c] <= thr[i] && myid < n_ref);
                        while (m) {
                            const int src = __ffs(m) - 1;
                            m &= m - 1;
                            const int c_l = __shfl_sync(SK_FULL, cnt[i][c], src);
                            const int ty_l = src >> 3, tx_l = src & 7;
                            const int qs = tile_query_slot(warp, ty_l, i);
                            const int id_l = idbase + tile_ref_slot(tx_l, c);
                            int nthr, nid;
                            list_insert<KC, int, true>(list_c, list_i, qs, c_l, id_l, lane, nthr, nid);
                            if (ty == ty_l) thr[i] = nthr;
                        }
                    }
                }
            }
        }
    }

    if constexpr (kRegLists) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const long long q = qtile * QTILE + tile_query_slot(warp, ty, i);
            if (q < n_q) {
#pragma unroll
                for (int e = 0; e < EPL; ++e) {
                    cand_idx[q * KC + tx * EPL + e] = li[i][e];
                    cand_cnt[q * KC + tx * EPL + e] = lk[i][e];
                }
            }
        }
        return;
    }
    for (int ql = 0; ql < 32; ++ql) {
        const int qs = warp * 32 + ql;
        const long long q = qtile * QTILE + qs;
        if (q >= n_q) break;
        if (lane < KC) {
            cand_idx[q * KC + lane] = list_i[qs * KC + lane];
            cand_cnt[q * KC + lane] = list_c[qs * KC + lane];
        }
    }
}

static size_t hamming_smem_bytes(int kc, int nstage, int wq_words) {
    const size_t lists = kc <= 16 ? 0 : (size_t)QTILE * kc * 8;  // <= 16: register lists
    return (size_t)nstage * HAM_STAGE * 4 + lists + (size_t)2 * nstage * 8 + (size_t)wq_words * 4;
}

template <int KC, bool WTD>
static cudaError_t launch_ham_kc(const uint32_t *qimg, const uint32_t *rimg, const uint32_t *wq,
                                 int n_chunks, int n_rtiles, long long n_q, int n_ref, int *cand_idx,
                                 int *cand_cnt, cudaStream_t st) {
    const int wq_words = WTD ? n_chunks * HAM_WC : 0;
    int nstage = 4;
    while (nstage > 2 && hamming_smem_bytes(KC, nstage, wq_words) > 227 * 1024) --nstage;
    const size_t smem = hamming_smem_bytes(KC, nstage, wq_words);
    if (smem > 227 * 1024) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(hamming_search_kernel<KC, WTD>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    const long long n_qtiles = (n_q + QTILE - 1) / QTILE;
    hamming_search_kernel<KC, WTD><<<(unsigned)n_qtiles, SEARCH_THREADS, smem, st>>>(
        qimg, rimg, wq, n_chunks, n_rtiles, nstage, n_q, n_ref, cand_idx, cand_cnt);
    return cudaGetLastError();
}

cudaError_t launch_hamming_search(const uint32_t *qimg, const uint32_t *rimg, const uint32_t *wq,
                                  int n_chunks, int n_rtiles, long long n_q, int n_ref, int kc,
                                  int *cand_idx, int *cand_cnt, cudaStream_t st) {
    if (n_q <= 0) return cudaSuccess;
    if (wq) {
        switch (kc) {
            case 16: return launch_ham_kc<16, true>(qimg, rimg, wq, n_chunks, n_rtiles, n_q, n_ref, cand_idx, cand_cnt, st);
            case 32: return launch_ham_kc<32, true>(qimg, rimg, wq, n_chunks, n_rtiles, n_q, n_ref, cand_idx, cand_cnt, st);
            default: return cudaErrorInvalidValue;
        }
    }
    switch (kc) {
        case 8: return launch_ham_kc<8, false>(qimg, rimg, nullptr, n_chunks, n_rtiles, n_q, n_ref, cand_idx, cand_cnt, st);
        case 16: return launch_ham_kc<16, false>(qimg, rimg, nullptr, n_chunks, n_rtiles, n_q, n_ref, cand_idx, cand_cnt, st);
        case 32: return launch_ham_kc<32, false>(qimg, rimg, nullptr, n_chunks, n_rtiles, n_q, n_ref, cand_idx, cand_cnt, st);
        default: return cudaErrorInvalidValue;
    }
}

// ---- counts -> float64 distances, then the common epilogue ------------------------------
__global__ void __launch_bounds__(256)
hamming_finish_kernel(const int *__restrict__ cand_idx, const int *__restrict__ cand_cnt, int kc,
                      const double *__restrict__ lut, long long n_q, FinishParams fp) {
    // (shuffle: the compiler then knows `warp` is warp-uniform and keeps what derives from it in uniform registers)
    const int warp = __shfl_sync(SK_FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const long long q = (long long)blockIdx.x * 8 + warp;
    if (q >= n_q) return;
    double d = SK_INF_D;
    int id = 0x7fffffff;
    if (lane < kc) {
        id = cand_idx[q * kc + lane];
        const int c = cand_cnt[q * kc + lane];
        if (id != 0x7fffffff) d = lut[c];
    }
    finish_query(fp, q, d, id, lane);
}

cudaError_t launch_hamming_finish(const int *cand_idx, const int *cand_cnt, int kc,
                                  const double *lut, long long n_q, const FinishParams &fp,
                                  cudaStream_t st) {
    if (n_q <= 0) return cudaSuccess;
    const long long grid = (n_q + 7) / 8;
    hamming_finish_kernel<<<(unsigned)grid, 256, 0, st>>>(cand_idx, cand_cnt, kc, lut, n_q, fp);
    return cudaGetLastError();
}

// ---- wide mode: exact 32-bit codes behind the 16-bit filter ---------------------------------
// A tree with more than 31743 distinct node IDs has no dense 16-bit coding.  The index then keeps
// exact u32 codes and runs the kernels above on their hashed image (wide mod 31743; 0xFFFFFFFF,
// "matches nothing", -> 31743).  Hashing only merges distinct codes, so a hashed mismatch count (or
// fixed-point sum) never exceeds the true one: every reference outside a filter list still has a
// true value >= the list's boundary, and hamming_refine_kernel certifies against that bound.
__global__ void __launch_bounds__(256)
hamming_hash_kernel(const uint32_t *__restrict__ wide, long long n, long long ldw, int n_trees,
                    uint16_t *__restrict__ codes) {
    const long long total = n * n_trees;
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < total; e += (long long)gridDim.x * 256) {
        const long long r = e / n_trees;
        const int t = (int)(e - r * n_trees);
        codes[e] = hamming_filter_code(wide[r * ldw + t]);
    }
}

cudaError_t launch_hamming_hash(const uint32_t *wide, long long n, long long ldw, int n_trees, uint16_t *codes,
                                cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    long long blocks = (n * n_trees + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    hamming_hash_kernel<<<(unsigned)blocks, 256, 0, st>>>(wide, n, ldw, n_trees, codes);
    return cudaGetLastError();
}

// ---- re-rank of the filter's candidates on the exact codes + certificate -------------------
// One warp per query, one filter candidate per lane; Code is the type of the exact codes (uint16_t:
// the searched codes themselves, uint32_t: wide mode).  The list's boundary is its largest (filter
// value, index).
// Unequal weights: the distance is SciPy's, the left-to-right float64 sum of w_t over the mismatching
// trees divided by the left-to-right sum of all w_t.  Every reference outside the list has a
// fixed-point sum >= the boundary's (bc), hence a true numerator >= scale * bc - err; the top k are
// final when the k-th exact numerator is below that.
// Equal weights (a.lut != null, wide mode only; 16-bit counts are exact and go to
// hamming_finish_kernel): the true mismatch counts, ranked by (count, index); every reference outside
// the list has a true (count, index) above the boundary, so the top k are final when the k-th is
// below it - a k-th tie with the boundary is decided by the index, exactly as the ranking decides it.
// Either way a list with an empty slot holds every reference.
template <class Code>
__global__ void __launch_bounds__(256)
hamming_refine_kernel(HammingRefineArgs a, FinishParams fp) {
    // (shuffle: the compiler then knows `warp` is warp-uniform and keeps what derives from it in uniform registers)
    const int warp = __shfl_sync(SK_FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const long long q = (long long)blockIdx.x * 8 + warp;
    if (q >= a.n_q) return;
    int id = 0x7fffffff, c = 0x7fffffff;
    if (lane < a.kc) {
        id = a.cand_idx[q * a.kc + lane];
        c = a.cand_cnt[q * a.kc + lane];
    }
    const bool valid = id != 0x7fffffff;
    const bool whole = __ballot_sync(SK_FULL, lane < a.kc && !valid) != 0;   // the list holds every reference
    // the list's boundary: its largest (filter value, index)
    int bc = valid ? c : -1, bi = valid ? id : -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const int oc = __shfl_xor_sync(SK_FULL, bc, o), oi = __shfl_xor_sync(SK_FULL, bi, o);
        if (pair_less<int>(bc, bi, oc, oi)) {
            bc = oc;
            bi = oi;
        }
    }
    const Code *qc = static_cast<const Code *>(a.qcodes) + q * a.ldq;
    const Code *rc = static_cast<const Code *>(a.rcodes) + (long long)(valid ? id : 0) * a.n_trees;
    const int kk = fp.k + (fp.exclude_self ? 1 : 0);
    bool ok;
    double d = SK_INF_D;
    if (a.lut) {
        int m = 0x7fffffff;
        if (valid) {
            m = 0;
            for (int t = 0; t < a.n_trees; ++t) m += qc[t] != rc[t];
        }
        warp_sort_pairs<int, 32>(m, id, lane);
        const int kc_ = __shfl_sync(SK_FULL, m, kk - 1), ki = __shfl_sync(SK_FULL, id, kk - 1);
        ok = whole || pair_less<int>(kc_, ki, bc, bi);
        if (id != 0x7fffffff) d = a.lut[m];
    } else {
        double num = SK_INF_D;
        if (valid) num = hamming_numerator(qc, rc, a.n_trees, a.w);
        warp_sort_pairs<double, 32>(num, id, lane);
        const double kth = __shfl_sync(SK_FULL, num, kk - 1);
        ok = whole || kth < a.scale * (double)bc - a.err;
        if (id != 0x7fffffff) d = num / a.wsum;
    }
    if (!ok) {
        if (lane == 0) {
            const int pos = atomicAdd(a.fb_count, 1);
            a.fb_list[pos] = (int)q;
        }
        return;
    }
    finish_query(fp, q, d, id, lane);
}

cudaError_t launch_hamming_refine(const HammingRefineArgs &a, bool wide, const FinishParams &fp, cudaStream_t st) {
    if (a.n_q <= 0) return cudaSuccess;
    const long long grid = (a.n_q + 7) / 8;
    if (wide)
        hamming_refine_kernel<uint32_t><<<(unsigned)grid, 256, 0, st>>>(a, fp);
    else
        hamming_refine_kernel<uint16_t><<<(unsigned)grid, 256, 0, st>>>(a, fp);
    return cudaGetLastError();
}

}  // namespace sk

// Shared device helpers for the sknnr_b200 kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <math.h>
#include <stdio.h>

#define SK_FULL 0xffffffffu
#define SK_INF_F __int_as_float(0x7f800000)
#define SK_INF_D __longlong_as_double(0x7ff0000000000000LL)

// Self-check build (python -m sknnr_b200._build --variant=checks -DSK_CHECKS): device-side bounds and
// protocol assertions in the kernels that manage shared memory by hand.  compute-sanitizer is closed
// on this pool, so the test suite is run against this build instead (profiles/r02_selfcheck.md).
#ifdef SK_CHECKS
#define SK_CHECK(cond)                                                                              \
    do {                                                                                            \
        if (!(cond)) {                                                                              \
            printf("SK_CHECK failed: %s (%s:%d) block %d thread %d\n", #cond, __FILE__, __LINE__,   \
                   (int)blockIdx.x, (int)threadIdx.x);                                              \
            __trap();                                                                               \
        }                                                                                           \
    } while (0)
#else
#define SK_CHECK(cond) ((void)0)
#endif

namespace sk {

constexpr int NCOMPUTE_WARPS = 12;
constexpr int QTILE = 32 * NCOMPUTE_WARPS;  // queries per CTA tile (32 per compute warp)
constexpr int RTILE = 64;       // reference plots per staged tile
constexpr int SEARCH_THREADS = NCOMPUTE_WARPS * 32;  // lane 0 of warp 0 also issues the TMA copies
constexpr int MAXK = 32;        // entries handled by one warp-wide sort
// tensor-core engine tile shape: M = 128 queries per MMA (2 M tiles per CTA), N = 128 plots
constexpr int TC_M = 128;
constexpr int TC_N = 128;

// A query value as float64, whatever the element type of the caller's matrix (kernels.h, with_x_type).
// Every integer of these types below 2^53 converts exactly; int64 beyond rounds to nearest, as NumPy's
// cast to float64 does - so the rest of a kernel sees the values the float64 path would.
__device__ __forceinline__ double x_to_f64(double v) { return v; }
__device__ __forceinline__ double x_to_f64(float v) { return (double)v; }
__device__ __forceinline__ double x_to_f64(uint8_t v) { return __uint2double_rn(v); }
__device__ __forceinline__ double x_to_f64(int16_t v) { return __int2double_rn(v); }
__device__ __forceinline__ double x_to_f64(uint16_t v) { return __uint2double_rn(v); }
__device__ __forceinline__ double x_to_f64(int32_t v) { return __int2double_rn(v); }
__device__ __forceinline__ double x_to_f64(long long v) { return __ll2double_rn(v); }

// ---------------------------------------------------------------------------------------
// mbarrier + 1-D TMA bulk copy (cp.async.bulk -> SASS UBLKCP)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// (the suspend-time hint lets the hardware park the warp until the phase completes instead of
// returning to the retry loop: waiting warps stop competing for issue slots)
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t addr = smem_u32(bar);
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(addr),
        "r"(parity), "r"(0x989680u)
        : "memory");
}
// variants taking a precomputed 32-bit shared-memory address (hot loops: no generic -> shared
// conversion per call)
__device__ __forceinline__ void mbar_wait_addr(uint32_t addr, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(addr),
        "r"(parity), "r"(0x989680u)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_addr(uint32_t addr) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(addr) : "memory");
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes,
                                         uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// round-to-nearest conversion to TF32 (10 explicit mantissa bits), result as FP32 bits
__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

// ---------------------------------------------------------------------------------------
// warp-wide bitonic sort of one (key, id) per lane, ascending by (key, id)
// ---------------------------------------------------------------------------------------
template <typename K>
__device__ __forceinline__ bool pair_less(K ka, int ia, K kb, int ib) {
    return (ka < kb) || (ka == kb && ia < ib);
}

template <typename K>
__device__ __forceinline__ K shfl_xor_any(K v, int m);
template <>
__device__ __forceinline__ float shfl_xor_any<float>(float v, int m) {
    return __shfl_xor_sync(SK_FULL, v, m);
}
template <>
__device__ __forceinline__ int shfl_xor_any<int>(int v, int m) {
    return __shfl_xor_sync(SK_FULL, v, m);
}
template <>
__device__ __forceinline__ double shfl_xor_any<double>(double v, int m) {
    return __shfl_xor_sync(SK_FULL, v, m);
}
template <>
__device__ __forceinline__ long long shfl_xor_any<long long>(long long v, int m) {
    return __shfl_xor_sync(SK_FULL, v, m);
}

// SIZE < 32 sorts every aligned group of SIZE lanes on its own (fewer network stages when only the
// first SIZE lanes hold entries)
template <typename K, int SIZE = 32>
__device__ __forceinline__ void warp_sort_pairs(K &key, int &id, int lane) {
#pragma unroll
    for (int size = 2; size <= SIZE; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            K ok = shfl_xor_any<K>(key, stride);
            int oi = __shfl_xor_sync(SK_FULL, id, stride);
            bool lower = (lane & stride) == 0;          // I hold the lower slot of the pair
            bool asc = (lane & size) == 0;              // this block sorts ascending
            bool other_less = pair_less<K>(ok, oi, key, id);
            // lower slot of an ascending block keeps the smaller element
            bool take = (lower == asc) ? other_less : !other_less && !(ok == key && oi == id);
            if (take) {
                key = ok;
                id = oi;
            }
        }
    }
}


// ---------------------------------------------------------------------------------------
// Sorted candidate lists in shared memory (one list of KC (key, id) entries per query,
// ascending).  Only the owning warp touches a query's list and lane L only ever touches
// slot L, so no barrier or atomic is needed.  Returns true when (key, id) was inserted and
// reports the list's new last entry.
//   LEX = false : accept only key <  last key            (float scores; exact ties are the
//                                                          certificate's business)
//   LEX = true  : accept (key, id) < (last key, last id)  (integer Hamming counts: the lowest
//                                                          index must win every tie)
// ---------------------------------------------------------------------------------------
template <typename K> __device__ __forceinline__ K key_sentinel();
template <> __device__ __forceinline__ float key_sentinel<float>() { return SK_INF_F; }
template <> __device__ __forceinline__ int key_sentinel<int>() { return 0x7fffffff; }

template <int KC, typename K, bool LEX>
__device__ __forceinline__ bool list_insert(K *list_k, int *list_i, int qs, K key, int id,
                                            int lane, K &last_k, int &last_i) {
    K ck = key_sentinel<K>();
    int ci = 0x7fffffff;
    if (lane < KC) {
        ck = list_k[qs * KC + lane];
        ci = list_i[qs * KC + lane];
    }
    const K cur_k = __shfl_sync(SK_FULL, ck, KC - 1);
    const int cur_i = __shfl_sync(SK_FULL, ci, KC - 1);
    const bool accept = LEX ? pair_less<K>(key, id, cur_k, cur_i) : (key < cur_k);
    if (!accept) {
        last_k = cur_k;
        last_i = cur_i;
        return false;
    }
    const unsigned lt = __ballot_sync(SK_FULL, pair_less<K>(ck, ci, key, id));
    const int pos = __popc(lt);
    const K pk = __shfl_up_sync(SK_FULL, ck, 1);
    const int pi = __shfl_up_sync(SK_FULL, ci, 1);
    if (lane == pos) {
        ck = key;
        ci = id;
    } else if (lane > pos) {
        ck = pk;
        ci = pi;
    }
    if (lane < KC) {
        list_k[qs * KC + lane] = ck;
        list_i[qs * KC + lane] = ci;
    }
    last_k = __shfl_sync(SK_FULL, ck, KC - 1);
    last_i = __shfl_sync(SK_FULL, ci, KC - 1);
    return true;
}

// thread <-> tile coordinates shared by the float and Hamming search kernels: lanes form a
// 4 (query groups, ty) x 8 (reference groups, tx) grid; a thread's 8 queries are two runs of
// 4 (LDS.128 each), likewise its 8 references.
__device__ __forceinline__ int tile_query_slot(int warp, int ty, int i) {
    return warp * 32 + ((i < 4) ? (ty * 4 + i) : (16 + ty * 4 + (i - 4)));
}
__device__ __forceinline__ int tile_ref_slot(int tx, int c) {
    return (c < 4) ? (tx * 4 + c) : (32 + tx * 4 + (c - 4));
}


// ---------------------------------------------------------------------------------------
// Register-resident candidate lists (KC = 8 * EPL <= 16).  The 8 lanes that share a query
// (same ty, tx = 0..7) hold its sorted list in registers: lane tx keeps list positions
// tx*EPL .. tx*EPL+EPL-1 of each of its 8 queries, so an insertion is a handful of width-8
// shuffles and the four lane groups of a warp insert into four different queries at once.
// No shared memory, no atomics, no barrier.
// ---------------------------------------------------------------------------------------
template <int EPL, typename K, bool LEX>
__device__ __forceinline__ void group_insert(K (&lk)[EPL], int (&li)[EPL], bool valid, K key,
                                             int id, int tx, int ty, K &thr_k) {
    // thr_k always mirrors the list's last key; only the tie-breaking (LEX) variant needs the
    // last index as well
    bool accept;
    if constexpr (LEX) {
        const int last_i = __shfl_sync(SK_FULL, li[EPL - 1], 7, 8);
        accept = valid && pair_less<K>(key, id, thr_k, last_i);
    } else {
        accept = valid && (key < thr_k);
    }
    int pos = 0;
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
        const unsigned b = __ballot_sync(SK_FULL, pair_less<K>(lk[e], li[e], key, id));
        pos += __popc((b >> (ty * 8)) & 0xffu);
    }
    const K prev_k = __shfl_up_sync(SK_FULL, lk[EPL - 1], 1, 8);
    const int prev_i = __shfl_up_sync(SK_FULL, li[EPL - 1], 1, 8);
    if (accept) {
#pragma unroll
        for (int e = EPL - 1; e >= 0; --e) {
            const int p = tx * EPL + e;
            const K sk = (e > 0) ? lk[e > 0 ? e - 1 : 0] : prev_k;
            const int si = (e > 0) ? li[e > 0 ? e - 1 : 0] : prev_i;
            if (p > pos) {
                lk[e] = sk;
                li[e] = si;
            } else if (p == pos) {
                lk[e] = key;
                li[e] = id;
            }
        }
    }
    thr_k = __shfl_sync(SK_FULL, lk[EPL - 1], 7, 8);
}

template <typename T>
__device__ __forceinline__ T select8(const T (&v)[8], int c) {
    const T a = (c & 1) ? v[1] : v[0];
    const T b = (c & 1) ? v[3] : v[2];
    const T d = (c & 1) ? v[5] : v[4];
    const T e = (c & 1) ? v[7] : v[6];
    const T ab = (c & 2) ? b : a;
    const T de = (c & 2) ? e : d;
    return (c & 4) ? de : ab;
}

// Drain the hits of one tile row (one of the thread's 8 queries): `sc` are this thread's 8
// scores for the row, `hm` the bit mask of those still below the threshold.  Every iteration
// each lane group elects its first lane with a pending hit and inserts that hit.
template <int EPL, typename K, bool LEX>
__device__ __forceinline__ void drain_row(const K (&sc)[8], unsigned hm, K (&lk)[EPL], int (&li)[EPL],
                                          K &thr, int idbase, int id_limit, int tx, int ty) {
    while (true) {
        const unsigned act = __ballot_sync(SK_FULL, hm != 0);
        if (act == 0) break;
        const unsigned g = (act >> (ty * 8)) & 0xffu;
        const bool gvalid = g != 0;
        const int ltx = gvalid ? (__ffs(g) - 1) : 0;
        const int c = (hm != 0) ? (__ffs(hm) - 1) : 0;
        const K my = select8<K>(sc, c);
        const int myid = idbase + tile_ref_slot(tx, c);
        const K key = __shfl_sync(SK_FULL, my, ltx, 8);
        const int id = __shfl_sync(SK_FULL, myid, ltx, 8);
        if (gvalid && tx == ltx) hm &= hm - 1;
        group_insert<EPL, K, LEX>(lk, li, gvalid && id < id_limit, key, id, tx, ty, thr);
    }
}

// ---------------------------------------------------------------------------------------
// finish_query: everything sknnr/sklearn do AFTER the k(+1) nearest are known.
//   lanes 0..kk-1 hold the exact neighbours sorted ascending by (dist, id).
//   * X=None self exclusion          $SP/sklearn/neighbors/_base.py:929-958
//   * deterministic re-ordering      ref:src/sknnr/_base.py:166-175
//   * outputs f64 / i64              ref:src/sknnr/_base.py:182
//   * weighted multi-output average  $SP/sklearn/neighbors/_regression.py:254-267 with
//     weights from _get_weights      $SP/sklearn/neighbors/_base.py:74-117
// One warp per query.
// ---------------------------------------------------------------------------------------
struct FinishParams {
    int k;              // neighbours to return
    int exclude_self;   // 1: lanes hold k+1 entries, drop the query itself
    int deterministic;
    double round_scale; // 10^decimals
    long long row_offset;
    double *out_dist;   // [n_q, k] or null
    long long *out_idx; // [n_q, k] or null
    int weights;        // SKNNR_W_*
    const double *y;    // [n_ref, n_out]
    int n_ref;          // guards the target gather against invalid ids (non-finite input)
    const int *row_map; // compacted launches: row_map[q] is the row of the original chunk
    int n_out;
    double *out_pred;   // [n_q, n_out]
};

template <int SIZE>
__device__ __forceinline__ void det_sort(double &key, long long &sec, double &dist, int lane) {
#pragma unroll
    for (int size = 2; size <= SIZE; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            double ok = __shfl_xor_sync(SK_FULL, key, stride);
            long long os = __shfl_xor_sync(SK_FULL, sec, stride);
            double od = __shfl_xor_sync(SK_FULL, dist, stride);
            bool lower = (lane & stride) == 0;
            bool asc = (lane & size) == 0;
            bool other_less = (ok < key) || (ok == key && os < sec);
            bool same = (ok == key && os == sec);
            bool take = (lower == asc) ? other_less : (!other_less && !same);
            if (take) {
                key = ok;
                sec = os;
                dist = od;
            }
        }
    }
}

// W = 32: one query per warp (`lane` 0..31).  W = 16: one query per half warp - every shuffle,
// vote and loop below stays inside the aligned 16-lane segment of the calling lane, `lane` is the
// lane within the segment, and `write` = false turns a segment into a silent passenger (its
// partner segment still needs the full warp in the shuffles).
template <int W>
__device__ __forceinline__ unsigned seg_ballot(bool pred) {
    const unsigned b = __ballot_sync(SK_FULL, pred);
    if constexpr (W == 32) {
        return b;
    } else {
        unsigned lane32;
        asm("mov.u32 %0, %%laneid;" : "=r"(lane32));
        return (b >> (lane32 & 16u)) & 0xffffu;
    }
}

template <int W>
__device__ __forceinline__ void finish_query_w(const FinishParams &p, long long q, double dist, int id,
                                               int lane, bool write) {
    if (p.row_map) q = p.row_map[q];
    const long long row = p.row_offset + q;
    int kk = p.k + (p.exclude_self ? 1 : 0);
    if (lane >= kk) {
        dist = SK_INF_D;
        id = 0x7fffffff;
    }
    if (p.exclude_self) {
        unsigned m = seg_ballot<W>(lane < kk && (long long)id == row);
        int pos = m ? (__ffs(m) - 1) : 0;
        double nd = __shfl_down_sync(SK_FULL, dist, 1, W);
        int ni = __shfl_down_sync(SK_FULL, id, 1, W);
        if (lane >= pos) {
            dist = nd;
            id = ni;
        }
        if (lane >= p.k) {
            dist = SK_INF_D;
            id = 0x7fffffff;
        }
    }
    if (p.deterministic) {
        // row_scale = max(rowmax, 1); rounded = rint(dist / row_scale * 10^dec) / 10^dec
        double rowmax = __shfl_sync(SK_FULL, dist, p.k - 1, W);  // ascending -> last is max
        double scale = fmax(rowmax, 1.0);
        // (lanes past k hold +inf: they divide 1.0 instead, which keeps the whole warp on the division's
        // fast path - an infinite operand sends all 32 lanes through the slow one)
        const double dsafe = (lane < p.k) ? dist : 1.0;
        double key = (lane < p.k) ? rint((dsafe / scale) * p.round_scale) / p.round_scale : SK_INF_D;
        long long diff = (long long)id - row;
        if (diff < 0) diff = -diff;
        // sort by (key, diff, id): fold (diff, id) into one 64-bit secondary key.  ids and
        // diffs are < 2^31 for any index this library accepts.
        long long sec = (lane < p.k) ? ((diff << 31) | (long long)id) : 0x7fffffffffffffffLL;
        // The lanes arrive sorted by (dist, id) and the key is monotone in dist, so the order can
        // only change inside a group of equal rounded keys: skip the network unless some
        // neighbouring pair is out of (key, sec) order (rare: ties to `decimals` digits).
        const double pk = __shfl_up_sync(SK_FULL, key, 1, W);
        const long long ps = __shfl_up_sync(SK_FULL, sec, 1, W);
        const bool out_of_order = lane > 0 && lane < p.k && (key < pk || (key == pk && sec < ps));
        // bitonic network on (key, sec) carrying dist; only the first k lanes hold entries, so the
        // network spans the next power of two >= k (sorting an ordered segment again is harmless)
        if (!__any_sync(SK_FULL, out_of_order)) {
        } else if (p.k <= 8)
            det_sort<8>(key, sec, dist, lane);
        else if (p.k <= 16)
            det_sort<16>(key, sec, dist, lane);
        else
            det_sort<32>(key, sec, dist, lane);
        id = (int)(sec & 0x7fffffffLL);
    }
    if (write && lane < p.k) {
        if (p.out_dist) p.out_dist[q * p.k + lane] = dist;
        if (p.out_idx) p.out_idx[q * p.k + lane] = (long long)id;
    }
    if (p.weights != 0 && p.out_pred != nullptr) {
        double w = 1.0;
        if (p.weights == 2) {
            unsigned zm = seg_ballot<W>(lane < p.k && dist == 0.0);
            if (zm)
                w = (dist == 0.0) ? 1.0 : 0.0;
            else
                w = 1.0 / ((lane < p.k) ? dist : 1.0);   // (padding lanes: fast-path operand, see above)
        }
        if (lane >= p.k) w = 0.0;
        double denom = 0.0;
        for (int c = 0; c < p.k; ++c) denom += __shfl_sync(SK_FULL, w, c, W);
        for (int j0 = 0; j0 < p.n_out; j0 += W) {
            int j = j0 + lane;
            double num = 0.0;
            for (int c = 0; c < p.k; ++c) {
                double wc = __shfl_sync(SK_FULL, w, c, W);
                int ic = __shfl_sync(SK_FULL, id, c, W);
                if (j < p.n_out && ic >= 0 && ic < p.n_ref) {
                    double yv = p.y[(long long)ic * p.n_out + j];
                    num = (p.weights == 1) ? (num + yv) : (num + yv * wc);
                }
            }
            if (write && j < p.n_out) {
                p.out_pred[q * p.n_out + j] = (p.weights == 1) ? (num / (double)p.k) : (num / denom);
            }
        }
    }
}

__device__ __forceinline__ void finish_query(const FinishParams &p, long long q, double dist,
                                             int id, int lane) {
    finish_query_w<32>(p, q, dist, id, lane, true);
}

// Numerator of SciPy's weighted Hamming distance: the left-to-right float64 sum of w_t over the
// trees whose codes differ ($SP/scipy/spatial/distance.py:1718-1723 -> cdist_hamming).  Code is
// uint16_t (dense node codes) or uint32_t (wide mode's exact codes).
template <class Code>
__device__ __forceinline__ double hamming_numerator(const Code *qc, const Code *rc, int n_trees,
                                                    const double *w) {
    double s = 0.0;
    for (int t = 0; t < n_trees; ++t)
        if (qc[t] != rc[t]) s = __dadd_rn(s, w[t]);
    return s;
}

}  // namespace sk

// Tensor-core engine of the fused distance + top-KC candidate search: tcgen05.mma (kind::f16, FP16
// operands, FP32 accumulators in TMEM), operands staged by 1-D TMA bulk copies, selection fused into
// the TMEM epilogue so the score matrix never leaves the SM.
//
// Same role as search_simt.cu (it replaces the dgemm + heap-test hot loop of scikit-learn's
// EuclideanArgKmin64, $SP/sklearn/metrics/_pairwise_distances_reduction/_argkmin.pyx.tp:401-510)
// but the contraction runs on the 5th-generation tensor cores.  FP16 operands carry 2^-11 relative
// error each (the 11-bit significand of TF32 at twice its MMA rate), so this kernel is only ever a
// FILTER: it returns (at most) the KC - 1 best references per stream by approximate score plus a
// threshold that every reference outside the lists is known to reach; refine.cu re-evaluates the
// survivors in float64 and proves (error bound eps_s ~ 2^-10) that nothing outside the lists can
// belong to the k nearest; rows it cannot certify come back to this kernel once (second pass: one
// stream of 15, every row from the threshold refine proved sufficient, `init_thr`), then go to the
// FP32 SIMT engine and, failing that, to the exhaustive float64 kernel.
//
// One CTA = 256 queries = two M=128 MMA tiles that share every 128-plot reference tile (N=128).  A
// "job" is one (reference tile, M tile) pair = K/16 tcgen05.mma into one of four 128-column TMEM
// accumulator slots; jobs run in (tile, M tile) order and job j uses slot j % 4, i.e. every M tile
// owns two slots and its MMAs run at most one job ahead of its scanners.  19 warps (ns = 2):
//   TMA producer (1 thread)   bulk copies (cp.async.bulk + mbarrier) of the query image once and of
//                    the reference tiles through an NSTAGE ring;
//   MMA issuers (one warp per M tile, warp-uniform loop, one elected lane)  wait "tile staged" and
//                    "slot drained", issue the job's tcgen05.mma, tcgen05.commit onto "slot ready"
//                    and (both issuers) "stage free";
//   16 scanner warps = (column stream p, M tile h, TMEM lane quarter): thread <-> (query, stream).
//                    Per job a warp waits "slot ready", reads its stream's 64 accumulator columns
//                    with one tcgen05.ld.x64, hands the slot back BEFORE reducing anything, then per
//                    32-column chunk: min3 tree over four octets -> one vote "did any lane beat its
//                    threshold".  If so, a ballot per octet picks the octets somebody hit, and every
//                    lane PARKS those of its octets whose minimum beats its threshold (8 raw scores +
//                    the first index) in its own pending queue in shared memory with predicated
//                    stores: straight-line code, no cross-lane traffic.  All scanner warps of the CTA
//                    RESOLVE their queues in the same jobs (every eighth, sooner when a queue is
//                    nearly full): tc_drain appends the values below the lane's threshold to the
//                    lane's candidate column, tc_compact (register bitonic network) keeps the entries
//                    below the KC-th best, lowers the threshold to it and - two streams - to the
//                    joint rank of both streams' published scores.  A score that cannot be stored
//                    lowers the threshold to itself instead (always valid, costs a certificate).
//   All role / slot / barrier values derive from a shuffled (provably warp-uniform) warp index and
//   live in uniform registers: the scanners have 96 vector registers, 64 of them hold a job.
//   (ns = 1: one stream of 16 candidates, 8 scanner warps of four chunks, for k (+1) <= 15.)
//
// Threshold seeding.  A streaming top-KC pays KC*ln(n_ref/KC) threshold hits per query, almost
// all of them while the threshold is still loose.  The kernel therefore first runs every
// `seed_stride`-th reference tile in a min-only mode that keeps 32 group minima per (query, stream)
// in the still unused candidate column; the KC-th smallest group minimum is an upper bound of the
// stream's KC-th best score (KC distinct references reach it), so the main pass starts with a
// threshold close to its final value: ~18 parked octets per stream instead of ~65 hits.
//
// The |r|^2 term is folded into the contraction: each operand gets three extra K elements holding
// (1,1,1) on the query side and a 3-way FP16 split of sigma^2 |r - mu|^2 on the reference side, so
// the accumulator is directly s = |r|^2 - 2 q.r.
//
// Operand layout (no swizzle, K-major "interleaved" canonical layout): 16-byte K chunks of 8 FP16
// values, [chunk][row][8]; core matrix = 8 rows x 16 B contiguous, SBO = 128 B between row
// groups, LBO = rows * 16 B between K chunks.  The images are pre-arranged in HBM in exactly
// this order, so a plain bulk copy stages them.
#include <cstdio>
#include "common.cuh"
#include "kernels.h"
#include "tc_common.cuh"

#include <type_traits>

namespace sk {

// MT M tiles (of 128 queries) per CTA; NS independent candidate streams per query: stream p owns
// columns [p * 128 / NS, (p + 1) * 128 / NS) of every reference tile and has its own scanner
// warps, candidate buffer and threshold; KCS candidates kept per stream, CAP buffer slots.
template <int MT_, int NS_, int CAP_, int CAPE_> struct TcCfg {
    static constexpr int MT = MT_, NS = NS_, CAP = CAP_, CAPE = CAPE_;
    static constexpr int QT = MT * TC_M;                  // queries per CTA
    static constexpr int EPI_WARPS = MT * 4 * NS;         // scanner warps: (stream, M tile, lane quarter)
    static constexpr int THREADS = (EPI_WARPS + MT + 1) * 32;  // + MT MMA issuer warps + TMA producer warp
    // slot stride of the candidate buffers: a power of two, so that a thread's slot count sits in the
    // high bits of its buffer offset (4 * column + count * LD * 4).  Threads work on their own
    // columns (bank = column mod 32, no conflicts); only the rare cooperative path, where a warp
    // writes into ONE column, serialises on a bank.
    static constexpr int LD = QT * NS;
    static constexpr int SORT = CAP <= 16 ? 16 : 32;      // width of the register sorting network
    static_assert(CAP <= SORT && CAP % 2 == 0, "candidate buffer shape");
    static constexpr int CH = 4 / NS;                     // 32-column chunks a scanner warp reads per job
};

// diagnostics of the debug instantiation (tc_debug bit 3): chunk visits, events, queued octets,
// drains, compactions, dropped octets / values - printed by the last CTA
__device__ unsigned long long g_tc_counters[8];

// rank (in the union of both streams' lists) of the score the joint threshold is set to: the k-th
// neighbour must clear it by the certificate's error margin, so it sits a few ranks above k
constexpr int TC_JOINT = 10;
// ... and the rank an index falls back to when too many of its rows fail rank TC_JOINT (api.cu, tc_wide_joint)
constexpr int TC_JOINT_WIDE = 12;

// ---- per-thread selection state (thread <-> (query, stream) = column `col` of every array) ----
//   candidates  buf_s / buf_i [CAP][LD]: unsorted (score, index) entries; the count lives in
//               pr = 4 * col + count * LD * 4 (LD * 4 is a power of two above 4 * col), the offset of
//               the next free score slot
//   pending     pq_v [CAPE][LD][8] f32 + pq_i [CAPE][LD]: octets of raw scores that contained a value
//               below the threshold, parked by the fast path and resolved later by the whole warp at
//               once (tc_drain); count in pqo = 32 * col + count * LD * 32
//   published   pub [KCP][LD]: the thread's KCP best scores (sorted) at its last compaction; the
//               partner stream of the same query reads them to form a joint threshold
// Dropping is always safe: a score that cannot be stored (queue or list full) lowers the thread's
// threshold to that score instead - every reference outside the list then still has a score >=
// the threshold, which is all the certificate needs (the row merely becomes harder to certify).

// Warp-wide compaction, thread-parallel: every thread reduces its OWN candidate column to the
// entries strictly below t = its KC-th smallest score and lowers its threshold to t (fewer than
// KC entries: t = +inf, nothing changes).  NS = 2: the sorted best scores are published and the
// threshold is further lowered to the KC-th smallest score of the union with the partner
// stream's published list (stale or torn reads only see older = larger scores: still an upper
// bound of the query's KC-th best).  Called by all 32 lanes.
template <int KC, int CAP, int LD, int NS, int J>
__device__ __forceinline__ ThrPr tc_compact(uint32_t bs0, uint32_t pub0, uint32_t c4, float thr, uint32_t pr) {
    static_assert(KC < CAP, "the buffer needs slack above KC");
    constexpr int SORT = CAP <= 16 ? 16 : 32;
    constexpr uint32_t IOFF = CAP * LD * 4, STEP = LD * 4;
    const uint32_t cs0 = bs0 + c4;
    const int cnt = (int)(pr / STEP);
    SK_CHECK((pr & (STEP - 1)) == c4 && cnt <= CAP);
    float s[SORT];
#pragma unroll
    for (int j = 0; j < SORT; ++j) s[j] = (j < CAP && j < cnt) ? lds_f32(cs0 + j * STEP) : SK_INF_F;
    sort_regs<SORT>(s);
    float t = s[KC - 1];
    if constexpr (NS == 2 && J < 2 * KC) {
        static_assert(LD == 512, "partner column = column ^ 256");
        const uint32_t mine = pub0 + c4, other = pub0 + (c4 ^ 1024u);
        float o[KC];
#pragma unroll
        for (int i = 0; i < KC; ++i) {
            st_shared_b32(mine + i * STEP, __float_as_uint(s[i]));
            o[i] = lds_f32(other + i * STEP);
        }
        const float joint = tc_union_rank<KC, J, SORT>(s, o);
        t = fminf(t, joint);
    }
    t = fminf(t, thr);
    uint32_t w = cs0;
#pragma unroll 4
    for (int j = 0; j < CAP; ++j) {
        const float v = lds_f32(cs0 + j * STEP);
        const int id = lds_s32(cs0 + IOFF + j * STEP);
        if (j < cnt && v < t) {
            st_shared_b32(w, __float_as_uint(v));
            st_shared_b32(w + IOFF, (uint32_t)id);
            w += STEP;
        }
    }
    ThrPr out;
    out.thr = t;
    out.pr = w - bs0;
    return out;
}

// Resolve the warp's pending octets, all lanes at once: iteration `it` takes every lane's it-th
// parked octet (lanes with fewer are passengers) and appends its values below the lane's
// threshold to the lane's candidate column, branch-free (every value is stored at the next free
// slot, the slot only advances for the values that qualify).  Compacts when a lane is down to
// its last two free slots; a third qualifying value of one octet is dropped (see above).
template <int KC, int CAP, int LD, int CAPE, int NS, int J, bool DBG>
__device__ __noinline__ ThrPr tc_drain(uint32_t bs0, uint32_t pqv0, uint32_t pqi0, uint32_t pub0, uint32_t c4,
                                       float thr, uint32_t pr, uint32_t pqo, int dbg) {
    constexpr uint32_t IOFF = CAP * LD * 4, STEP = LD * 4, ES = LD * 32;
    constexpr uint32_t FULL = (CAP - 2) * STEP, LAST = (CAP - 1) * STEP;
    const int n_me = (int)(pqo / ES);
    SK_CHECK((pqo & (ES - 1)) == 8u * c4 && n_me <= CAPE);
    const int n_it = __reduce_max_sync(SK_FULL, n_me);
    for (int it = 0; it < n_it; ++it) {   // warp-uniform
        const bool act = it < n_me;
        if (__any_sync(SK_FULL, act && pr >= FULL)) {
            if (DBG && (dbg & 8) && (threadIdx.x & 31) == 0) atomicAdd(&g_tc_counters[4], 1ull);
            const ThrPr c = tc_compact<KC, CAP, LD, NS, J>(bs0, pub0, c4, thr, pr);
            thr = c.thr;
            pr = c.pr;
        }
        const uint32_t va = pqv0 + 8u * c4 + (uint32_t)it * ES;
        const float4 x = lds_f32x4(va), y = lds_f32x4(va + 16);
        const int id = lds_s32(pqi0 + c4 + (uint32_t)it * STEP);
        SK_CHECK(!act || (id >= 0 && (id & 7) == 0));
        SK_CHECK(pr <= LAST + c4);
        const float vv[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            st_shared_b32(bs0 + pr, __float_as_uint(vv[j]));
            st_shared_b32(bs0 + pr + IOFF, (uint32_t)(id + j));
            const bool q = act && vv[j] < thr;
            if (q) {
                if (pr < LAST) pr += STEP;
                else thr = fminf(thr, vv[j]);
            }
        }
    }
    ThrPr out;
    out.thr = thr;
    out.pr = pr;
    out.n_it = n_it;
    return out;
}

// One 32-column chunk of the main pass.  `r` holds this thread's scores against references
// idb .. idb+31.  Fast path: min3 tree over four octets + one vote.  On a hit anywhere in the warp
// every lane parks the octets whose minimum beats its threshold (predicated stores, no branch, no
// cross-lane traffic); what the values are is sorted out later by tc_drain.
template <int LD, int CAPE, bool DBG>
__device__ __forceinline__ void tc_chunk(const uint32_t (&r)[32], int idb, uint32_t pqv0, uint32_t pqi0, float &thr,
                                         uint32_t &pqo, int dbg) {
    constexpr uint32_t ES = LD * 32, PQ_END = CAPE * ES;
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
    float g[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) {
        const float *w = v + 8 * o;
        g[o] = fminf(fminf(fminf(fminf(w[0], w[1]), w[2]), fminf(fminf(w[3], w[4]), w[5])), fminf(w[6], w[7]));
    }
    const float m = fminf(fminf(fminf(g[0], g[1]), g[2]), g[3]);
    const bool hit = m < thr;
    if constexpr (DBG) {
        const unsigned hits = __ballot_sync(SK_FULL, hit);
        if ((dbg & 8) && (threadIdx.x & 31) == 0) {
            atomicAdd(&g_tc_counters[0], 1ull);
            if (hits) atomicAdd(&g_tc_counters[1], 1ull);
        }
        if (hits == 0u) return;
        if (dbg & 1) return;   // timing experiment: skip the hit path (results are wrong)
    } else {
        if (!__any_sync(SK_FULL, hit)) return;   // vote straight into a predicate
    }
    // which octets hold a hit somewhere in the warp (votes against the threshold on entry: it only
    // falls inside, so a vote can only be a false alarm); octets without one are skipped, branch uniform
    unsigned ov[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) ov[o] = __ballot_sync(SK_FULL, g[o] < thr);
#pragma unroll
    for (int o = 0; o < 4; ++o) {
        if (ov[o] == 0u) continue;
        const bool p = g[o] < thr;
        const bool room = pqo < PQ_END;
        SK_CHECK(pqo < PQ_END + ES);
        tc_dump8(p && room, pqv0 + pqo, pqi0 + (pqo >> 3), v + 8 * o, idb + 8 * o);
        if (p && !room) thr = fminf(thr, g[o]);
        if (p && room) pqo += ES;
        if (DBG && (dbg & 8) && p) atomicAdd(&g_tc_counters[room ? 2 : 5], 1ull);
    }
}

// Epilogue of one job (reference tile x this warp's M tile): the warp's CH chunks of 32 columns
// are all read into registers first and the accumulator slot is handed back to the MMA issuer
// BEFORE any of them is reduced, so the MMAs of the slot's next job overlap the reduction and a
// slow hit path never holds TMEM.
template <int CH, class F>
__device__ __forceinline__ void tc_epi_job(uint32_t (&R)[CH][32], uint32_t tcol, uint32_t afull_addr,
                                           uint32_t parity, uint32_t aempty_addr, int lane, F &&proc) {
    mbar_wait_addr(afull_addr, parity);
    tc_fence_after();
    if constexpr (CH == 2) {
        tmem_ld64_issue(tcol, R[0], R[1]);
    } else if constexpr (CH == 4) {
        tmem_ld64_issue(tcol, R[0], R[1]);
        tmem_ld64_issue(tcol + 64, R[2], R[3]);
    } else {
        uint32_t dep = 0;
#pragma unroll
        for (int c = 0; c < CH; ++c) tmem_ld32_issue(tcol + 32 * c, R[c], dep);
    }
#pragma unroll
    for (int c = 0; c < CH; ++c) tmem_ld_wait(R[c]);
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive_addr(aempty_addr);
    if constexpr (CH >= 1) proc(R[0], std::integral_constant<int, 0>{});
    if constexpr (CH >= 2) proc(R[1], std::integral_constant<int, 1>{});
    if constexpr (CH >= 3) proc(R[2], std::integral_constant<int, 2>{});
    if constexpr (CH >= 4) proc(R[3], std::integral_constant<int, 3>{});
}

// (register budget: the register file is allocated per 4 warps, so the 18-warp dual-stream CTA
// gets 65536 / (20 * 32) = 102 -> 96 registers per thread and the 10-warp one 168)
template <int KC, int MT, int NS, int CAP, int CAPE, int J, bool DBG>
__global__ void __launch_bounds__(TcCfg<MT, NS, CAP, CAPE>::THREADS, 1)
search_tc_kernel(const __half *__restrict__ qimg, const __half *__restrict__ rimg, int kc_tot,
                 int n_rtiles, int nstage, int n_seed, int seed_stride, long long n_q,
                 int *__restrict__ cand_idx, float *__restrict__ cand_thr, int dbg,
                 const float *__restrict__ init_thr, const int *__restrict__ n_rows_dev) {
    using Cfg = TcCfg<MT, NS, CAP, CAPE>;
    if (n_rows_dev) {   // compacted launch (second pass): only the first *n_rows_dev rows exist
        const long long n_dev = *n_rows_dev;
        if ((long long)blockIdx.x * Cfg::QT >= n_dev) return;
        n_q = min(n_q, n_dev);
    }
    constexpr int LD = Cfg::LD, EPI_WARPS = Cfg::EPI_WARPS;
    constexpr bool JOINT = NS == 2 && J < 2 * KC;     // J = 2 KC: every stream keeps its own KC-th best
    constexpr int KCP = JOINT ? KC : 0;               // published scores per thread
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const uint32_t a_bytes = (uint32_t)kc_tot * TC_M * TC_ROWB;  // one 128-query operand image
    const uint32_t b_bytes = (uint32_t)kc_tot * TC_N * TC_ROWB;  // one 128-plot operand image
    unsigned char *Qs = smem_raw;                                // MT operand images
    unsigned char *Rs = Qs + MT * a_bytes;                       // nstage operand images
    float *buf_s = reinterpret_cast<float *>(Rs + (size_t)nstage * b_bytes);   // candidates [CAP][LD]
    int *buf_i = reinterpret_cast<int *>(buf_s + CAP * LD);
    float *pq_v = reinterpret_cast<float *>(buf_i + CAP * LD);                 // pending [CAPE][LD][8]
    int *pq_i = reinterpret_cast<int *>(pq_v + CAPE * LD * 8);                 //         [CAPE][LD]
    float *pub = reinterpret_cast<float *>(pq_i + CAPE * LD);                  // published [KCP][LD]
    uint64_t *full = reinterpret_cast<uint64_t *>(pub + KCP * LD);             // (8-byte aligned: LD * 4 % 8 == 0)
    uint64_t *empty = full + nstage;
    uint64_t *afull = empty + nstage;       // [4] accumulator slot ready
    uint64_t *aempty = afull + TC_SLOTS;    // [4] accumulator slot drained
    uint64_t *qbar = aempty + TC_SLOTS;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(qbar + 1);

    // the shuffle tells the compiler that `warp` (and every role / slot / address value derived from
    // it) is warp-uniform: those live in uniform registers, not in the scanners' 96 vector registers
    const int warp = __shfl_sync(SK_FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < nstage; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], MT);   // one tcgen05.commit per MMA issuer
        }
        for (int a = 0; a < TC_SLOTS; ++a) {
            mbar_init(&afull[a], 1);
            mbar_init(&aempty[a], 4 * NS);  // the scanner warps of the M tile that used the slot
        }
        mbar_init(qbar, 1);
        fence_mbar_init();
    }
    if (warp == EPI_WARPS) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const long long qtile = blockIdx.x;
    const int ksteps = kc_tot >> 1;  // MMA K = 16 FP16 = two 16-byte chunks
    const int n_seq = n_seed + n_rtiles;  // sampled tiles (seeding), then every tile

    if (warp == EPI_WARPS + MT) {
        // ======================= TMA producer (one thread) =======================
        // No divisions, no descriptor rebuilds in these two single-thread loops: each of their
        // instructions is on the critical path of the tensor pipe.
        if (lane == 0) {
            mbar_expect_tx(qbar, MT * a_bytes);
            bulk_g2s(Qs, (const unsigned char *)qimg + (size_t)qtile * MT * a_bytes, MT * a_bytes, qbar);
            int sn = 0;
            uint32_t wrap_par = 1;   // parity of (uses of the slot so far - 1); first pass: no wait
            bool wrapped = false;
            const unsigned char *rbase = (const unsigned char *)rimg;
            for (int tn = 0; tn < n_seq; ++tn) {
                if (wrapped) mbar_wait(&empty[sn], wrap_par);
                const int tile = tn < n_seed ? tn * seed_stride : tn - n_seed;
                if (DBG && (dbg & 4) && wrapped) {
                    mbar_arrive(&full[sn]);   // timing experiment: reuse the stale tile, no L2 traffic
                } else {
                    mbar_expect_tx(&full[sn], b_bytes);
                    bulk_g2s(Rs + (size_t)sn * b_bytes, rbase + (size_t)tile * b_bytes, b_bytes, &full[sn]);
                }
                if (++sn == nstage) {
                    sn = 0;
                    wrap_par = wrapped ? (wrap_par ^ 1u) : 0u;
                    wrapped = true;
                }
            }
        }
        __syncwarp();
    } else if (warp >= EPI_WARPS) {
        // ======================= MMA issuers: one warp per M tile =======================
        // Issuing is effectively synchronous (the thread gets the next tcgen05.mma out at the
        // rate the tensor pipe retires them), and barrier waits + bookkeeping cost a lone warp
        // another ~300 cycles per job during which ITS MMAs are not being queued; with one issuer
        // per M tile the other issuer's MMAs fill that gap.
        // The whole warp runs the loop in lock step (uniform control flow keeps descriptors and
        // counters in uniform registers); one elected lane issues the tcgen05 instructions.
        const int h = warp - EPI_WARPS;
        mbar_wait(qbar, 0);
        const uint32_t a_lbo = TC_M * TC_ROWB, b_lbo = TC_N * TC_ROWB;
        // descriptor = {hi: SBO = 128 B, version 1; lo: start address >> 4 | LBO >> 4 << 16}; moving
        // to the next K step (two 16-byte chunks) or operand image only adds to the address field
        const uint64_t desc_hi = (uint64_t)((128u >> 4) | (1u << 14)) << 32;
        const uint32_t a_lo0 = (((smem_u32(Qs) + h * a_bytes) >> 4) & 0x3fffu) | (((a_lbo >> 4) & 0x3fffu) << 16);
        const uint32_t b_lo0 = ((smem_u32(Rs) >> 4) & 0x3fffu) | (((b_lbo >> 4) & 0x3fffu) << 16);
        const uint32_t a_kstep = (2 * a_lbo) >> 4, b_kstep = (2 * b_lbo) >> 4;
        const uint32_t b_img = b_bytes >> 4;
        int s = 0;
        uint32_t full_par = 0, b_lo_s = b_lo0;
        for (int t = 0; t < n_seq; ++t) {
            const int j = t * MT + h;                    // this issuer's job on tile t
            const uint32_t sl = (uint32_t)j & (TC_SLOTS - 1);
            mbar_wait(&full[s], full_par);
            if (j >= TC_SLOTS) mbar_wait(&aempty[sl], (uint32_t)(((j >> 2) - 1) & 1));
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + sl * TC_N;
            SK_CHECK(s >= 0 && s < nstage && sl < TC_SLOTS);
            if (elect_one()) {
                if (DBG && (dbg & 16)) {   // timing experiment: the job's MMAs issued twice (same result)
                    uint32_t a2 = a_lo0, b2 = b_lo_s;
                    tc_mma_f16(d_tmem, desc_hi | a2, desc_hi | b2, TC_IDESC, 0u);
                    for (int ks = 1; ks < ksteps; ++ks) {
                        a2 += a_kstep;
                        b2 += b_kstep;
                        tc_mma_f16(d_tmem, desc_hi | a2, desc_hi | b2, TC_IDESC, 1u);
                    }
                }
                uint32_t a_lo = a_lo0, b_lo = b_lo_s;
                tc_mma_f16(d_tmem, desc_hi | a_lo, desc_hi | b_lo, TC_IDESC, 0u);
#pragma unroll 4
                for (int ks = 1; ks < ksteps; ++ks) {
                    a_lo += a_kstep;
                    b_lo += b_kstep;
                    tc_mma_f16(d_tmem, desc_hi | a_lo, desc_hi | b_lo, TC_IDESC, 1u);
                }
                tc_commit(&afull[sl]);   // accumulators of job j complete
                tc_commit(&empty[s]);    // one of the MT arrivals that free the smem slot
            }
            __syncwarp();
            b_lo_s += b_img;
            if (++s == nstage) {
                s = 0;
                full_par ^= 1u;
                b_lo_s = b_lo0;
            }
        }
    } else {
        // ======================= epilogue: thread <-> (query, stream) =======================
        // warp = (stream p, M tile h, lane quarter); every warp takes part in every job of its M
        // tile and reads the stream's CH chunks of the 128 accumulator columns
        constexpr int CH = Cfg::CH;
        const int col = threadIdx.x;          // candidate buffer column of this (query, stream)
        const int p = warp / (MT * 4);
        const int h = (warp >> 2) % MT;
        const int qslot = h * TC_M + (warp & 3) * 32 + lane;   // query within the CTA = TMEM lane of M tile h
        const uint32_t tlane = tmem_base + (((uint32_t)((warp & 3) * 32)) << 16) + (uint32_t)(p * CH * 32);
        // Second pass over the rows the first one could not certify: every row comes with a threshold
        // just above what its top k needs (refine.cu, retry_threshold), so the lists end up holding
        // exactly the references below it and nothing is dropped on the way.  No seeding then; rows
        // past the end take -inf (no hits).
        float thr = SK_INF_F;
        if (init_thr) {
            const long long q_me = qtile * Cfg::QT + qslot;
            thr = q_me < n_q ? init_thr[q_me] : -SK_INF_F;
        }
        uint32_t R[CH][32];
        int t = 0;                            // position in the tile sequence; this warp's job = t * MT + h
        const uint32_t afull_a0 = smem_u32(afull), aempty_a0 = smem_u32(aempty);

        // shared-window addresses of the selection arrays, derived from the dynamic array's own shared
        // address (no generic pointer round trip): uniform registers
        const uint32_t bs0 = smem_u32(smem_raw) + MT * a_bytes + (uint32_t)nstage * b_bytes;
        const uint32_t pqv0 = bs0 + 2u * CAP * LD * 4u, pqi0 = pqv0 + (uint32_t)CAPE * LD * 32u;
        const uint32_t pub0 = pqi0 + (uint32_t)CAPE * LD * 4u;
        const uint32_t c4 = 4u * (uint32_t)col;
        if constexpr (KCP > 0) {
#pragma unroll
            for (int i = 0; i < KCP; ++i) st_shared_b32(pub0 + c4 + i * (LD * 4), __float_as_uint(SK_INF_F));
        }

        // ---- seeding pass: group minima over the sampled tiles ----
        // (the 32 running minima live in the still unused candidate buffer column: slots of
        // buf_s, then of buf_i; chunk c of the n-th sampled tile feeds group (CH * n + c) % 32)
        if (n_seed > 0) {
            static_assert(2 * CAP >= TC_GROUPS, "group minima are parked in the candidate buffers");
            float *gcol = buf_s + col;
#pragma unroll
            for (int g = 0; g < TC_GROUPS; ++g) gcol[g * LD] = SK_INF_F;   // buf_i follows buf_s
            // (few sampled tiles: a group is an octet of columns instead of a chunk, so that even a
            // reference set of a few hundred plots fills more than KC groups)
            const bool fine = n_seed * CH < TC_GROUPS;
            for (; t < n_seed; ++t) {
                const int j = t * MT + h, sl = j & (TC_SLOTS - 1);
                const int g0 = (t * CH) & (TC_GROUPS - 1);
                tc_epi_job<CH>(R, tlane + (uint32_t)(sl * TC_N), afull_a0 + 8u * sl, (uint32_t)((j >> 2) & 1),
                               aempty_a0 + 8u * sl, lane,
                               [&](const uint32_t (&r)[32], auto ic) {
                                   constexpr int c = decltype(ic)::value;
                                   if (!fine) {
                                       float *g = gcol + (g0 + c) * LD;
                                       *g = fminf(*g, tc_min32(r));
                                   } else {
#pragma unroll
                                       for (int o = 0; o < 4; ++o) {
                                           float m = __uint_as_float(r[8 * o]);
#pragma unroll
                                           for (int e = 1; e < 8; ++e) m = fminf(m, __uint_as_float(r[8 * o + e]));
                                           float *g = gcol + (((t * CH + c) * 4 + o) & (TC_GROUPS - 1)) * LD;
                                           *g = fminf(*g, m);
                                       }
                                   }
                               });
            }
            float gm[TC_GROUPS];
#pragma unroll
            for (int g = 0; g < TC_GROUPS; ++g) gm[g] = gcol[g * LD];
            sort_regs<TC_GROUPS>(gm);
            thr = gm[KC - 1];
            if constexpr (KCP > 0) {
                // joint seed: the KC-th smallest group minimum of BOTH streams of the query.  The two
                // warps of a (M tile, lane quarter) pair meet on a named barrier so that each sees
                // the other's minima.
#pragma unroll
                for (int i = 0; i < KC; ++i) st_shared_b32(pub0 + c4 + i * (LD * 4), __float_as_uint(gm[i]));
                asm volatile("bar.sync %0, 64;" ::"r"(1 + (warp & (MT * 4 - 1))) : "memory");
                float o[KC];
#pragma unroll
                for (int i = 0; i < KC; ++i) o[i] = lds_f32(pub0 + (c4 ^ 1024u) + i * (LD * 4));
                const float joint = tc_union_rank<KC, J, TC_GROUPS>(gm, o);
                thr = fminf(thr, joint);
            }
        }

        // ---- main pass ----
        constexpr uint32_t ES = LD * 32;
        uint32_t pr = c4;            // offset of this thread's next free candidate slot (4 * col + count * LD * 4)
        uint32_t pqo = 8u * c4;      // offset of its next free pending-queue entry (32 * col + count * LD * 32)
        int since_drain = 1;   // countdown to an extra resolution (the first one right after the first job)
        const int early_tiles = max(64, n_rtiles >> 3);
        for (; t < n_seq; ++t) {
            const int j = t * MT + h, sl = j & (TC_SLOTS - 1);
            const int idb = (t - n_seed) * TC_N + p * CH * 32;   // warp-uniform, like t and p
            tc_epi_job<CH>(R, tlane + (uint32_t)(sl * TC_N), afull_a0 + 8u * sl, (uint32_t)((j >> 2) & 1),
                           aempty_a0 + 8u * sl, lane,
                           [&](const uint32_t (&r)[32], auto ic) {
                               constexpr int c = decltype(ic)::value;
                               tc_chunk<LD, CAPE, DBG>(r, idb + c * 32, pqv0, pqi0, thr, pqo, dbg);
                           });
            // Every scanner warp of the CTA resolves its queues in the SAME jobs: a slot is only handed
            // back when all eight warps of its M tile have read it, so a long operation costs the
            // whole M tile its duration - once per period when the warps take it together, almost
            // every job when each warp takes it whenever its own queues fill up (measured: 32.5 ->
            // 30.1 ms per 4M rows).  A lane whose queue fills up inside a period drops octets, which
            // only lowers its threshold.
            constexpr int DRAIN_EVERY = 8;   // jobs between two scheduled resolutions (a power of two)
            // The schedule is global (job number modulo the period).  On top of it a warp whose queues
            // were (nearly) full at its last resolution comes back after one or two jobs: early in the
            // pass and on small reference sets the thresholds are loose and a full period would overflow
            // the queues (dropped octets lower thresholds and cost certificates).  A countdown, not a
            // vote: the fast path pays one uniform compare.
            bool now;
            if constexpr (CAPE >= 4 && NS == 2) {
                now = (((t - n_seed) & (DRAIN_EVERY - 1)) == DRAIN_EVERY - 1) | (--since_drain == 0);
                // (the first tiles of the main pass - all of them on a small reference set - also look
                // at the queues themselves: there the thresholds move fast and a warp-wide vote per job,
                // 3.6 % of the kernel when it is paid on every tile, buys 5 - 10x fewer uncertified rows)
                if ((t - n_seed) < early_tiles) now |= __any_sync(SK_FULL, pqo >= (uint32_t)(CAPE - 1) * ES);
            } else {
                // (one stream of four chunks per job, or queues of two octets: a period would overflow
                // the queues, so a lane with a parked octet makes its warp resolve at once)
                now = __any_sync(SK_FULL, pqo >= ES);
            }
            if (now) {
                if (DBG && (dbg & 8) && lane == 0) atomicAdd(&g_tc_counters[3], 1ull);
                if (DBG && (dbg & 32)) {   // timing experiment: park but never resolve (results are wrong)
                    pqo = 8u * c4;
                    since_drain = -1;
                    continue;
                }
                const ThrPr d = tc_drain<KC, CAP, LD, CAPE, NS, J, DBG>(bs0, pqv0, pqi0, pub0, c4, thr, pr, pqo, dbg);
                thr = d.thr;
                pr = d.pr;
                pqo = 8u * c4;
                since_drain = d.n_it >= CAPE - 1 ? 1 : (d.n_it >= CAPE - 2 ? 2 : -1);
            }
        }

        // ---- flush the queue, final compaction, then every thread writes the candidates of its
        //      (query, stream) ----
        {
            const ThrPr d = tc_drain<KC, CAP, LD, CAPE, NS, J, DBG>(bs0, pqv0, pqi0, pub0, c4, thr, pr, pqo, dbg);
            const ThrPr c = tc_compact<KC, CAP, LD, NS, J>(bs0, pub0, c4, d.thr, d.pr);
            thr = c.thr;
            pr = c.pr;
        }
        const int cnt = (int)(pr / (uint32_t)(LD * 4));
        SK_CHECK(cnt < KC && cnt <= 16 / NS);
        const long long q = qtile * Cfg::QT + qslot;
        if (q < n_q) {
            constexpr int KOUT = 16 / NS;   // list slots per stream in the output (unused ones hold -1)
            int4 *dst = reinterpret_cast<int4 *>(cand_idx + (q * NS + p) * KOUT);
#pragma unroll
            for (int jj = 0; jj < KOUT; jj += 4) {
                int4 v;
                v.x = (jj + 0 < cnt) ? buf_i[(jj + 0) * LD + col] : -1;
                v.y = (jj + 1 < cnt) ? buf_i[(jj + 1) * LD + col] : -1;
                v.z = (jj + 2 < cnt) ? buf_i[(jj + 2) * LD + col] : -1;
                v.w = (jj + 3 < cnt) ? buf_i[(jj + 3) * LD + col] : -1;
                dst[jj / 4] = v;
            }
            cand_thr[q * NS + p] = thr;  // +inf only when the list holds every reference of the stream
        }
    }

    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == EPI_WARPS) tmem_dealloc(tmem_base, 512);
    if (DBG && (dbg & 8) && blockIdx.x == gridDim.x - 1 && threadIdx.x == 0)
        printf("tc counters (up to the last CTA): chunks %llu events %llu queued %llu drains %llu compactions %llu dropped %llu\n",
               g_tc_counters[0], g_tc_counters[1], g_tc_counters[2], g_tc_counters[3], g_tc_counters[4],
               g_tc_counters[5]);
}

int g_tc_debug = 0;  // timing experiments only (set through the "tc_debug" option)

// Two stream layouts:
//   ns = 2: two streams of 8 candidates (CAP 16) per query, 16 scanner warps -- k (+1) <= 7
//   ns = 1: one stream of 16 candidates (CAP 32), 8 scanner warps            -- k (+1) <= 15
// (a list keeps the entries strictly below its KC-th best score, i.e. KC - 1 candidates)
// and two pending-queue depths (4, or 2 when the operand images leave less shared memory).
static constexpr int TC_MT = 2;

size_t search_tc_smem_bytes(int kc_tot, int nstage, int ns, int cape) {
    const size_t a = (size_t)kc_tot * TC_M * TC_ROWB, b = (size_t)kc_tot * TC_N * TC_ROWB;
    // (published scores only exist while the joint threshold is on: two streams, d' <= 45)
    const size_t ld = (size_t)TC_MT * TC_M * ns, cap = ns == 2 ? 16 : 32, kcp = (ns == 2 && kc_tot <= 6) ? 8 : 0;
    return TC_MT * a + nstage * b + ld * 4 * (2 * cap + (size_t)cape * 9 + kcp) +
           (size_t)(2 * nstage + 2 * TC_SLOTS + 1) * 8 + 16;
}

// ring stages (low byte) and pending-queue depth (next byte) for this contraction depth; 0: the
// shape does not fit the engine
int search_tc_pick_config(int kc_tot) {
    const int capes[2] = {4, 2};
    for (int ci = 0; ci < 2; ++ci)
        for (int s = 4; s >= 2; --s)
            if (search_tc_smem_bytes(kc_tot, s, 2, capes[ci]) <= 227 * 1024 &&
                search_tc_smem_bytes(kc_tot, s, 1, capes[ci]) <= 227 * 1024)
                return s | (capes[ci] << 8);
    return 0;
}

// sampled tiles of the seeding pass (0 = no seeding: too few references for it to pay)
// The kernel starts with infinite thresholds, and a pass that starts cold parks far more octets than
// its queues hold (dropped octets cost certificates), so the sample is never switched off: small
// reference sets are pre-scanned completely (they are cheap), mid-sized ones every second tile.
int search_tc_seed_stride(int n_rtiles, int seed_stride) {
    if (seed_stride <= 0) seed_stride = 4;
    if (n_rtiles < 64) return 1;
    if (n_rtiles < 192) return seed_stride < 2 ? seed_stride : 2;
    return seed_stride;
}
int search_tc_seed_tiles(int n_rtiles, int seed_stride) {
    const int st = search_tc_seed_stride(n_rtiles, seed_stride);
    return (n_rtiles + st - 1) / st;
}

template <int KC, int MT, int NS, int CAP, int CAPE, int J, bool DBG>
static cudaError_t launch_tc_dbg(const __half *qimg, const __half *rimg, int kc_tot, int n_rtiles, int nstage,
                                 int seed_stride, long long n_q, int *cand_idx, float *cand_thr,
                                 const float *init_thr, const int *n_rows_dev, cudaStream_t st) {
    using Cfg = TcCfg<MT, NS, CAP, CAPE>;
    const size_t smem = search_tc_smem_bytes(kc_tot, nstage, NS, CAPE);
    cudaError_t e = cudaFuncSetAttribute(search_tc_kernel<KC, MT, NS, CAP, CAPE, J, DBG>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    const long long n_qtiles = (n_q + Cfg::QT - 1) / Cfg::QT;
    const int n_seed = init_thr ? 0 : search_tc_seed_tiles(n_rtiles, seed_stride);
    search_tc_kernel<KC, MT, NS, CAP, CAPE, J, DBG><<<(unsigned)n_qtiles, Cfg::THREADS, smem, st>>>(
        qimg, rimg, kc_tot, n_rtiles, nstage, n_seed, search_tc_seed_stride(n_rtiles, seed_stride), n_q, cand_idx,
        cand_thr, g_tc_debug, init_thr, n_rows_dev);
    return cudaGetLastError();
}

template <int KC, int MT, int NS, int CAP>
static cudaError_t launch_tc(const __half *qimg, const __half *rimg, int kc_tot, int n_rtiles, int nstage,
                             int cape, int seed_stride, int wide_joint, long long n_q, int *cand_idx, float *cand_thr,
                             const float *init_thr, const int *n_rows_dev, cudaStream_t st) {
    // rank of the joint threshold: the certificate's margin grows with the contraction depth
    // (eps * (|q|^2 + max|r|^2)), so deep spaces keep the streams' own KC-th best (rank 2 KC = off)
    constexpr int JLO = NS == 2 ? TC_JOINT : 1, JMID = NS == 2 ? TC_JOINT_WIDE : 1, JHI = NS == 2 ? 2 * KC : 1;
    const bool deep = kc_tot > 6;   // more than 48 FP16 elements, i.e. d' > 45 (search_tc_smem_bytes knows the same rule)
#define SK_TC_GO(CAPE_, J_, DBG_)                                                                                  \
    return launch_tc_dbg<KC, MT, NS, CAP, CAPE_, J_, DBG_>(qimg, rimg, kc_tot, n_rtiles, nstage, seed_stride, n_q, \
                                                           cand_idx, cand_thr, init_thr, n_rows_dev, st)
    // the timing-experiment hooks ("tc_debug") live in a separate instantiation: none of their
    // tests is compiled into the product kernel
    if (g_tc_debug && cape == 4 && !deep) SK_TC_GO(4, JLO, true);
    if (cape == 4 && !deep && NS == 2 && wide_joint) SK_TC_GO(4, JMID, false);
    if (cape == 4 && !deep) SK_TC_GO(4, JLO, false);
    if (cape == 4) SK_TC_GO(4, JHI, false);
    if (cape == 2) SK_TC_GO(2, JHI, false);
#undef SK_TC_GO
    return cudaErrorInvalidValue;
}

// cand_idx [n_q][16] (ns lists of 16 / ns entries), cand_thr [n_q][ns]; `config` from search_tc_pick_config
cudaError_t launch_search_tc(const __half *qimg, const __half *rimg, int kc_tot, int n_rtiles,
                             long long n_q, int ns, int config, int seed_stride, int wide_joint, int *cand_idx,
                             float *cand_thr, const float *init_thr, const int *n_rows_dev, cudaStream_t st) {
    if (n_q <= 0) return cudaSuccess;
    const int nstage = config & 0xff, cape = (config >> 8) & 0xff;
    if (ns == 2)
        return launch_tc<8, TC_MT, 2, 16>(qimg, rimg, kc_tot, n_rtiles, nstage, cape, seed_stride, wide_joint, n_q,
                                          cand_idx, cand_thr, init_thr, n_rows_dev, st);
    if (ns == 1)
        return launch_tc<16, TC_MT, 1, 32>(qimg, rimg, kc_tot, n_rtiles, nstage, cape, seed_stride, 0, n_q,
                                           cand_idx, cand_thr, init_thr, n_rows_dev, st);
    return cudaErrorInvalidValue;
}

}  // namespace sk

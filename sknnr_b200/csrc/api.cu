// extern "C" entry points of libsknnr_b200.so (see include/sknnr_b200.h for the contract and
// the reference seams each call replaces).  Host-side orchestration only: fitted-state upload,
// chunked streaming of query rows through project -> search -> refine -> exact(fallback), and
// copies.  No CPU compute path exists here: every call needs a CUDA device.
#include "../../include/sknnr_b200.h"
#include "common.cuh"
#include "kernels.h"

#include <algorithm>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <deque>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <chrono>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <vector>

using namespace sk;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}

#define CK(expr)                                                                              \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            char _b[512];                                                                     \
            snprintf(_b, sizeof(_b), "CUDA error %s at %s:%d: %s", cudaGetErrorName(_e),      \
                     __FILE__, __LINE__, cudaGetErrorString(_e));                             \
            return fail(_e == cudaErrorMemoryAllocation ? SKNNR_ENOMEM : SKNNR_ECUDA, _b);    \
        }                                                                                     \
    } while (0)

struct Options {
    int64_t engine = SKNNR_ENGINE_AUTO;
    int64_t chunk_rows = 1 << 20;
    int64_t timing = 0;
    int64_t kc = 16; // minimum candidate-list length of the float search (0 = smallest that fits k+1)
    int64_t tc_streams = 0;     // tensor engine: candidate streams per query (0 = automatic, else 1 or 2)
    int64_t host_slots = 8;     // a host-buffer call keeps min(4, host_slots) chunks in flight (1..8)
    int64_t tc_seed_stride = 4; // tensor engine: pre-scan every n-th reference tile to seed thresholds (0 = default)
    int64_t stage_rows = 1 << 19; // rows per chunk of a call whose buffers are pageable
} g_opt;

// ---- host staging of pageable buffers -----------------------------------------------------
// cudaMemcpyAsync on pageable memory goes through the driver's own bounce buffer on the calling
// thread at a fraction of the PCIe rate.  Callers of the estimators hand over ordinary NumPy arrays,
// so the library stages them itself: a few worker threads copy a chunk into (out of) page-locked
// slot buffers while the GPU works on the previous chunks.
class HostPool {
    std::vector<std::thread> th_;
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<std::function<void()>> q_;

    void worker() {
        for (;;) {
            std::function<void()> f;
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return !q_.empty(); });
                f = std::move(q_.front());
                q_.pop_front();
            }
            f();
        }
    }

public:
    explicit HostPool(int n) {
        for (int i = 0; i < n; ++i) {
            th_.emplace_back([this] { worker(); });
            th_.back().detach();   // the pool lives until the process exits
        }
    }
    int size() const { return (int)th_.size(); }
    static HostPool &get() {
        static HostPool *pool = [] {
            const unsigned hw = std::thread::hardware_concurrency();
            const int n = (int)std::min(16u, std::max(2u, hw * 3 / 4));
            return new HostPool(n - 1);   // the calling thread takes a share as well
        }();
        return *pool;
    }
    // run f(i) for i in [0, n) on the workers and the caller; returns when all are done
    void parallel_for(int n, const std::function<void(int)> &f) {
        if (n <= 0) return;
        struct Sync {
            std::mutex m;
            std::condition_variable cv;
            int left;
        } sy;
        sy.left = n - 1;
        for (int i = 1; i < n; ++i) {
            std::lock_guard<std::mutex> lk(m_);
            q_.emplace_back([&sy, &f, i] {
                f(i);
                std::lock_guard<std::mutex> l2(sy.m);
                if (--sy.left == 0) sy.cv.notify_one();
            });
            cv_.notify_one();
        }
        f(0);
        std::unique_lock<std::mutex> lk(sy.m);
        sy.cv.wait(lk, [&] { return sy.left == 0; });
    }
};

// A staging copy is written once and read next by the DMA engine (or by the caller much later):
// streaming stores keep it out of the cache and spare the read-for-ownership of every destination
// line, a third of the copy's memory traffic (8 threads on the build host: 21 -> 27 GB/s).
void stream_copy(unsigned char *d, const unsigned char *s, size_t n) {
#if defined(__SSE2__)
    if (n >= (256u << 10)) {
        while (n && ((uintptr_t)d & 15)) { *d++ = *s++; --n; }
        for (size_t i = n / 64; i; --i, s += 64, d += 64) {
            const __m128i a = _mm_loadu_si128((const __m128i *)s), b = _mm_loadu_si128((const __m128i *)(s + 16));
            const __m128i c = _mm_loadu_si128((const __m128i *)(s + 32)), e = _mm_loadu_si128((const __m128i *)(s + 48));
            _mm_stream_si128((__m128i *)d, a);
            _mm_stream_si128((__m128i *)(d + 16), b);
            _mm_stream_si128((__m128i *)(d + 32), c);
            _mm_stream_si128((__m128i *)(d + 48), e);
        }
        _mm_sfence();
        n %= 64;
    }
#endif
    memcpy(d, s, n);
}

// rows x row_bytes from src (row stride src_ld bytes) to dst (row stride dst_ld bytes), split over the pool
void parallel_copy_rows(void *dst, size_t dst_ld, const void *src, size_t src_ld, size_t row_bytes, int64_t rows) {
    if (rows <= 0 || row_bytes == 0) return;
    HostPool &pool = HostPool::get();
    const size_t total = (size_t)rows * row_bytes;
    int parts = (int)std::min<size_t>((size_t)pool.size() + 1, std::max<size_t>(1, total >> 21));   // >= 2 MB each
    const int64_t per = (rows + parts - 1) / parts;
    pool.parallel_for(parts, [&](int i) {
        const int64_t r0 = (int64_t)i * per, r1 = std::min(rows, r0 + per);
        if (r0 >= r1) return;
        unsigned char *d = (unsigned char *)dst + (size_t)r0 * dst_ld;
        const unsigned char *sp = (const unsigned char *)src + (size_t)r0 * src_ld;
        if (dst_ld == row_bytes && src_ld == row_bytes) {
            stream_copy(d, sp, (size_t)(r1 - r0) * row_bytes);
        } else {
            for (int64_t r = r0; r < r1; ++r, d += dst_ld, sp += src_ld) memcpy(d, sp, row_bytes);
        }
    });
}

void parallel_copy_flat(void *dst, const void *src, size_t bytes) {
    const size_t piece = 1 << 20;
    parallel_copy_rows(dst, piece, src, piece, piece, (int64_t)(bytes / piece));
    if (bytes % piece) memcpy((unsigned char *)dst + bytes / piece * piece, (const unsigned char *)src + bytes / piece * piece, bytes % piece);
}

// true for ordinary (not page-locked, not device, not managed) host memory
bool is_pageable(const void *p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

// true for device (or managed) memory: such an X needs no copy in, such outputs are reached by a
// device-to-device (possibly peer, over NVLink) copy
bool is_device_ptr(const void *p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

template <typename T>
struct PinBuf {
    T *p = nullptr;
    size_t cap = 0;  // elements
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaHostAlloc((void **)&p, n * sizeof(T), cudaHostAllocDefault);
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

int round_up(int v, int m) { return (v + m - 1) / m * m; }

int pick_kc(int kk, int slack) {
    const int need = kk + slack;
    if (need <= 8) return 8;
    if (need <= 16) return 16;
    if (need <= 32) return 32;
    return 0;
}

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;  // elements
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, n * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// per-chunk device buffers + the stream the chunk runs on
struct Slot {
    cudaStream_t stream = nullptr;
    // the cascade's tail (SIMT re-search + exhaustive search of uncertified rows) runs on its own
    // stream so that a handful of slow CTAs overlap the next chunk's first stage
    cudaStream_t tail_stream = nullptr;
    cudaEvent_t ev_stage1 = nullptr, ev_tail = nullptr;
    bool tail_pending = false;
    DevBuf<unsigned char> x;       // staged query rows (host callers)
    DevBuf<double> z64;
    DevBuf<float> qimg;
    DevBuf<__half> qimg_tc;        // tensor-core engine query image (FP16)
    DevBuf<double> z64c;           // compacted rows of the cascade's second stage
    DevBuf<int> fb2;               // second-stage failures: [0] = count, [1..] = list
    DevBuf<int> fbm;               // failures of the tensor engine's second pass (stage 1b), same layout
    DevBuf<float> fb_thr;          // second-pass thresholds of the first-stage failures (order of fb's list)
    DevBuf<uint16_t> codes;        // node codes produced by the device forest walk
    DevBuf<int> ids32;             // node IDs of sknnr_forest_apply
    DevBuf<uint32_t> qimg_h;       // Hamming query image
    DevBuf<int> cand_idx;
    DevBuf<float> cand_thr;
    DevBuf<int> cand_cnt;
    DevBuf<int> fb;                // [0] = count, [1..] = list
    DevBuf<double> o_dist;
    DevBuf<long long> o_idx;
    DevBuf<double> o_pred;
    // raster front end: compacted feature rows, pixel -> row map, group offsets, band-major results
    DevBuf<unsigned char> xc;
    DevBuf<int> r_pos, r_cnt;
    DevBuf<double> r_dist, r_pred;
    DevBuf<long long> r_idx;
    int *h_cnt = nullptr;          // pinned: valid pixels of the block in flight
    cudaEvent_t ev_cnt = nullptr;
    std::vector<cudaEvent_t> evs;  // pooled (start, stop) pairs around the search kernels
    size_t ev_used = 0;            // events handed out since the last harvest
    int *h_fb = nullptr;           // pinned: [0] first-stage, [1] second-stage failures, [2] non-finite flag, [3] rows of the FP32 stage
    bool fb_pending = false;
    long long rows_in_flight = 0;
    DevBuf<int> nonfinite;         // [0] != 0: a query value of the chunk in flight is NaN / inf
    bool flag_pending = false;
    // the slot's scratch stays in use until ev_last (the D2H of a host-buffer call's chunk, the end of a
    // device-pointer call's chunk on the caller's stream: such calls are not synchronised)
    cudaEvent_t ev_last = nullptr;
    bool last_pending = false;
    // host-buffer calls: the chunk's input has arrived / its first stage is through
    cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    // page-locked staging of pageable caller buffers (one chunk in, one chunk out) and the copy-out
    // that is still owed to the caller once the slot's stream has drained
    PinBuf<unsigned char> h_x, h_dist, h_idx, h_pred;
    struct CopyOut { void *dst; const void *src; size_t bytes; };
    std::vector<CopyOut> owed;
    void release() {
        x.release(); z64.release(); qimg.release(); qimg_tc.release(); z64c.release(); fb2.release(); fbm.release(); fb_thr.release();
        codes.release(); ids32.release(); qimg_h.release(); cand_idx.release();
        cand_thr.release(); cand_cnt.release(); fb.release(); o_dist.release();
        o_idx.release(); o_pred.release();
        xc.release(); r_pos.release(); r_cnt.release(); r_dist.release(); r_pred.release(); r_idx.release();
        if (h_cnt) cudaFreeHost(h_cnt);
        if (ev_cnt) cudaEventDestroy(ev_cnt);
        h_cnt = nullptr; ev_cnt = nullptr;
        for (auto e : evs) cudaEventDestroy(e);
        evs.clear();
        ev_used = 0;
        if (h_fb) cudaFreeHost(h_fb);
        nonfinite.release();
        h_x.release(); h_dist.release(); h_idx.release(); h_pred.release();
        owed.clear();
        if (ev_last) cudaEventDestroy(ev_last);
        ev_last = nullptr; last_pending = false; flag_pending = false;
        if (ev_in) cudaEventDestroy(ev_in);
        if (ev_out) cudaEventDestroy(ev_out);
        ev_in = ev_out = nullptr;
        if (stream) cudaStreamDestroy(stream);
        if (tail_stream) cudaStreamDestroy(tail_stream);
        if (ev_stage1) cudaEventDestroy(ev_stage1);
        if (ev_tail) cudaEventDestroy(ev_tail);
        tail_stream = nullptr; ev_stage1 = ev_tail = nullptr; tail_pending = false;
        h_fb = nullptr; stream = nullptr;
    }
    // record a timing event on `st` (pairs: even = start, odd = stop)
    cudaError_t mark(cudaStream_t st) {
        if (ev_used == evs.size()) {
            cudaEvent_t e;
            cudaError_t rc = cudaEventCreate(&e);
            if (rc != cudaSuccess) return rc;
            evs.push_back(e);
        }
        return cudaEventRecord(evs[ev_used++], st);
    }
};

struct IndexBase {
    int device = 0;
    int64_t n_ref = 0;
    int n_out = 0;
    double *d_y = nullptr;
    std::mutex lock;
    // chunks rotate through the slots (own stream + buffers each): H2D of one chunk, kernels of
    // another and D2H of a third overlap; a device-pointer call alternates the first two
    static constexpr int kSlots = 8;
    Slot slots[kSlots];
    int exact_grid = 0;
    sknnr_stats stats{};
    int n_sm = 148;
    bool spread_tail = true;   // run_chunk: deal the second stage's rows out over all SMs (set per chunk by the caller)
    long long n_exact_rows = 0;     // rows that reached the exhaustive kernel (last call)
    long long n_simt_rows = 0;      // rows that reached the FP32 stage after the tensor engine (last call)
    long long chunk_rows_seen = 0;  // adaptive engine choice: rows / cost-weighted first-stage failures seen
    long long chunk_fb_seen = 0;
    long long chunk_fail_seen = 0;  // plain count of first-pass failures (same window)
    bool tc_wide_joint = false;     // tensor engine, two streams: joint threshold at rank 12 instead of 10
    // Host-buffer calls run as a three-stage pipeline over a few slots of buffers: every chunk's input
    // goes through ONE in-order H2D stream, its kernels through ONE compute stream (the slots' tail
    // streams take the uncertified rows, as in a device-pointer call), its results through ONE D2H
    // stream.  (One stream per chunk, round 1's layout, left it to the driver how eight streams share
    // its hardware queues: traced on this pool, chunk c only started once chunk c - 2 was through.)
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr, host_compute = nullptr;

    int init_common(int dev, const double *y, int64_t nref, int nout) {
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
            return fail(SKNNR_ENODEV, "no CUDA device: sknnr_b200 has no CPU fallback");
        if (dev < 0 || dev >= count) return fail(SKNNR_EINVAL, "bad device ordinal");
        device = dev;
        n_ref = nref;
        n_out = nout;
        CK(cudaSetDevice(device));
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10)
            return fail(SKNNR_ENODEV, "sknnr_b200 kernels are built for sm_100a (B200) only");
        n_sm = prop.multiProcessorCount;
        if (y && nout > 0) {
            CK(cudaMalloc(&d_y, (size_t)nref * nout * sizeof(double)));
            CK(cudaMemcpy(d_y, y, (size_t)nref * nout * sizeof(double), cudaMemcpyHostToDevice));
        }
        int prio_lo = 0, prio_hi = 0;
        CK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CK(cudaStreamCreateWithFlags(&host_compute, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&h2d_stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&d2h_stream, cudaStreamNonBlocking));
        for (auto &s : slots) {
            CK(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
            // (the tail's few CTAs go ahead of the thousands the next chunk's first stage has queued:
            // the chunk's results are complete, and its slot free, a whole first stage earlier)
            CK(cudaStreamCreateWithPriority(&s.tail_stream, cudaStreamNonBlocking, prio_hi));
            CK(cudaEventCreateWithFlags(&s.ev_stage1, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&s.ev_tail, cudaEventDisableTiming));
            CK(cudaHostAlloc((void **)&s.h_fb, 4 * sizeof(int), cudaHostAllocDefault));
            s.h_fb[0] = s.h_fb[1] = s.h_fb[2] = s.h_fb[3] = 0;
            CK(s.nonfinite.reserve(1));
            CK(cudaEventCreateWithFlags(&s.ev_last, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&s.ev_in, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&s.ev_out, cudaEventDisableTiming));
            CK(cudaHostAlloc((void **)&s.h_cnt, sizeof(int), cudaHostAllocDefault));
            CK(cudaEventCreateWithFlags(&s.ev_cnt, cudaEventDisableTiming));
        }
        return SKNNR_OK;
    }
    void release_common() {
        cudaSetDevice(device);
        for (auto &s : slots) s.release();
        for (cudaStream_t *st : {&host_compute, &h2d_stream, &d2h_stream}) {
            if (*st) cudaStreamDestroy(*st);
            *st = nullptr;
        }
        exact_scr.release(); exact_big.release();
        if (ev_exact) cudaEventDestroy(ev_exact);
        ev_exact = nullptr;
        if (d_y) cudaFree(d_y);
        d_y = nullptr;
    }
    // collect timing / fallback count of the chunk that last ran on this slot
    void harvest(Slot &s) {
        for (size_t i = 0; i + 1 < s.ev_used; i += 2) {
            float ms = 0.f;
            if (cudaEventSynchronize(s.evs[i + 1]) == cudaSuccess &&
                cudaEventElapsedTime(&ms, s.evs[i], s.evs[i + 1]) == cudaSuccess)
                stats.search_ms += ms;
        }
        s.ev_used = 0;
        if (s.fb_pending) {
            stats.n_fallback += s.h_fb[0];
            n_exact_rows += s.h_fb[1];
            n_simt_rows += s.h_fb[3];
            chunk_rows_seen += s.rows_in_flight;
            // what a first-pass failure costs: about a third of a row's first pass when the second pass
            // certifies it, twenty times that when it goes on to the FP32 engine
            chunk_fb_seen += s.h_fb[3] * 6LL + s.h_fb[0];
            chunk_fail_seen += s.h_fb[0];
            // the two-stream layout's joint threshold sits at rank 10 of the query's candidates; data whose
            // neighbours crowd inside the FP16 error margin (few features, many plots) fail that more
            // than the second pass is worth: such an index moves to rank 12 for good
            if (chunk_rows_seen >= 4096 && chunk_fail_seen * 25 > chunk_rows_seen) tc_wide_joint = true;
            s.fb_pending = false;
        }
        if (s.flag_pending) {
            if (s.h_fb[2] != 0) saw_nonfinite = true;
            s.flag_pending = false;
        }
    }
    // The exhaustive kernel's scratch ([CTAs][n_ref] distances, + the big-k selection arrays) exists
    // once per index: its launches (cascade tails of different slots) are chained through ev_exact.
    DevBuf<double> exact_scr, exact_big;
    // CTAs of an exhaustive launch: two per SM, fewer when n_ref is so large that their distance
    // rows would exceed 1 GB of scratch
    int exact_ctas(int64_t rows) const {
        const int64_t by_mem = std::max<int64_t>(1, (int64_t)(1 << 30) / (8 * std::max<int64_t>(n_ref, 1)));
        return (int)std::max<int64_t>(0, std::min<int64_t>({rows, (int64_t)n_sm * 2, by_mem}));
    }
    cudaEvent_t ev_exact = nullptr;
    bool exact_used = false;
    cudaError_t launch_exact_chained(ExactArgs &ea, const FinishParams &fp, int kk, cudaStream_t st) {
        if (ea.grid <= 0) return cudaSuccess;
        cudaError_t e = exact_scr.reserve((size_t)exact_ctas(1 << 30) * (size_t)ea.n_ref);   // (a growing reserve frees the
        if (e != cudaSuccess) return e;                                         //  old block: cudaFree waits)
        ea.scratch = exact_scr.p;
        ea.big = nullptr;
        if (kk > MAXK) {
            e = exact_big.reserve((size_t)ea.grid * 4 * (size_t)kk);
            if (e != cudaSuccess) return e;
            ea.big = exact_big.p;
        }
        if (!ev_exact) {
            e = cudaEventCreateWithFlags(&ev_exact, cudaEventDisableTiming);
            if (e != cudaSuccess) return e;
        }
        if (exact_used) {
            e = cudaStreamWaitEvent(st, ev_exact, 0);
            if (e != cudaSuccess) return e;
        }
        e = launch_exact(ea, fp, st);
        if (e != cudaSuccess) return e;
        exact_used = true;
        return cudaEventRecord(ev_exact, st);
    }
    bool saw_nonfinite = false;   // some query value of the last call was NaN / inf
    // Wait until everything the slot was last used for is complete (its own stream, its tail, a
    // device-pointer caller's stream), hand the staged results of that chunk to the caller and
    // collect its counters.  After this the slot's buffers are free.
    cudaError_t finish_slot(Slot &s) {
        cudaError_t e = cudaStreamSynchronize(s.stream);
        if (e == cudaSuccess && s.tail_pending) e = cudaEventSynchronize(s.ev_tail);
        if (e == cudaSuccess && s.last_pending) e = cudaEventSynchronize(s.ev_last);
        s.tail_pending = false;
        s.last_pending = false;
        if (e == cudaSuccess)
            for (auto &c : s.owed) parallel_copy_flat(c.dst, c.src, c.bytes);
        s.owed.clear();
        harvest(s);
        return e;
    }
    // error path: nothing of this call may still be reading or writing caller memory when it returns
    void quiesce() {
        for (cudaStream_t st : {h2d_stream, host_compute}) if (st) cudaStreamSynchronize(st);
        for (auto &s : slots) {
            cudaStreamSynchronize(s.stream);
            if (s.tail_stream) cudaStreamSynchronize(s.tail_stream);
            if (s.last_pending) cudaEventSynchronize(s.ev_last);
            s.tail_pending = s.last_pending = s.fb_pending = s.flag_pending = false;
            s.owed.clear();
            s.ev_used = 0;
        }
        if (d2h_stream) cudaStreamSynchronize(d2h_stream);
        cudaGetLastError();
    }
};

// a device-pointer call lends the caller's stream to a slot for one chunk; the slot's own stream
// comes back whatever way the scope is left
struct StreamLoan {
    Slot &s;
    cudaStream_t saved;
    StreamLoan(Slot &slot, cudaStream_t st, bool lend) : s(slot), saved(slot.stream) {
        if (lend) s.stream = st;
    }
    ~StreamLoan() { s.stream = saved; }
};
// leaves the handle quiescent when a call fails half way through its chunks
struct CallGuard {
    IndexBase *ix;
    cudaStream_t user;
    bool ok = false;
    CallGuard(IndexBase *i, cudaStream_t u) : ix(i), user(u) {}
    ~CallGuard() {
        if (ok) return;
        if (user) cudaStreamSynchronize(user);
        ix->quiesce();
    }
};

// Rows of chunk `ci` of a call with `left` rows still to go.  Host buffers: the first chunk's H2D copy
// and the last chunk's D2H copy cannot overlap any kernel, so the stream of chunks ramps up (1/4, 1/2,
// 1, ...) and down (..., 1/2, 1/4 of `chunk`); the remainder rides in the chunk before the ramp down.
int64_t next_chunk_rows(int ci, int64_t left, int64_t chunk, bool ramp) {
    if (!ramp) return std::min(chunk, left);
    const int64_t q4 = chunk / 4;
    if (ci == 0) return q4;
    if (ci == 1) return 2 * q4;
    if (left > chunk + 3 * q4) return chunk;
    if (left > 3 * q4) {                                  // leaves 1/2 + 1/4 for the last two
        const int64_t rows = left - 3 * q4;
        return rows < q4 ? rows + 2 * q4 : rows;          // (a sliver rides with the half chunk instead)
    }
    if (left > q4) return left - q4;
    return left;
}
bool ramp_applies(bool dev_ptrs, int64_t n_q, int64_t chunk) { return !dev_ptrs && n_q >= 4 * chunk && chunk % 1024 == 0; }

int check_query_args(int64_t n_ref, int n_out, int64_t n_q, int k, uint32_t flags, int weights,
                     const void *X, const double *out_pred, int &kk) {
    const bool excl = flags & SKNNR_EXCLUDE_SELF;
    kk = k + (excl ? 1 : 0);
    if (k < 1) return fail(SKNNR_EINVAL, "k must be >= 1");
    if (kk > n_ref)
        return fail(SKNNR_EINVAL, excl ? "Expected n_neighbors < n_samples_fit"
                                       : "Expected n_neighbors <= n_samples_fit");
    if (excl && X != nullptr) return fail(SKNNR_EINVAL, "X must be NULL with SKNNR_EXCLUDE_SELF");
    if (!excl && (X == nullptr || n_q < 0)) return fail(SKNNR_EINVAL, "X is NULL");
    if (weights != SKNNR_W_NONE) {
        if (weights != SKNNR_W_UNIFORM && weights != SKNNR_W_DISTANCE)
            return fail(SKNNR_EINVAL, "bad weights mode");
        if (out_pred == nullptr || n_out <= 0)
            return fail(SKNNR_EINVAL, "prediction requested but no targets / output buffer");
    }
    return SKNNR_OK;
}

}  // namespace

// =========================================================================================
struct sknnr_index : IndexBase {
    int d_in = 0, d_out = 0, dpad = 0;
    double *d_ref64 = nullptr, *d_center = nullptr, *d_scale = nullptr, *d_proj = nullptr,
           *d_mu = nullptr;
    int metric = SKNNR_METRIC_EUCLIDEAN;
    float *d_rimg = nullptr;
    int n_rtiles = 0;
    double r2max = 0.0;            // max_j |ref_j - mu|^2; Manhattan / Chebyshev: max_j |ref_j - mu| in that norm
    bool simt_ok = true;           // the FP32 image can serve as a filter (Manhattan / Chebyshev: no plot overflows it)
    __half *d_rimg_tc = nullptr;   // tensor-core engine reference image (FP16)
    int n_rtiles_tc = 0, kc_tot = 0, tc_nstage = 0;
    double tc_sigma = 1.0;         // power-of-two scale of both tensor-engine images
    bool tensor_ok = false;        // shape fits the tensor engine
    // too many uncertified rows: the SIMT engine is the better first stage.  Decided per stream layout
    // (index = candidate streams per query: k (+1) <= 7 and larger k behave differently), from the
    // chunks of host-buffer calls with that layout only.
    bool tensor_demoted[3] = {false, false, false};
    int ns_in_use = 2;
};

struct sknnr_hamming_index : IndexBase {
    int n_trees = 0, n_chunks = 0, n_rtiles = 0;
    uint16_t *d_rcodes = nullptr;
    uint32_t *d_rimg = nullptr;
    double *d_w = nullptr, *d_lut = nullptr;
    double wsum = 0.0;
    bool uniform = true;
    // unequal weights: 16-bit fixed-point filter weights (two trees per word, like the code images)
    uint32_t *d_wq = nullptr;
    double wq_scale = 0.0, wq_err = 0.0;
    bool wq_ok = false;
};

struct sknnr_forest {
    int device = 0;
    int n_trees = 0, n_features = 0;
    long long n_nodes = 0;
    ForestNode *d_nodes = nullptr;
    int *d_roots = nullptr;
    std::mutex lock;
    cudaStream_t stream = nullptr;
    DevBuf<unsigned char> x;
    DevBuf<int> ids;
};

extern "C" {

const char *sknnr_last_error(void) { return g_err.c_str(); }
int sknnr_abi_version(void) { return SKNNR_ABI_VERSION; }

int sknnr_device_count(int *count) {
    if (!count) return fail(SKNNR_EINVAL, "count is NULL");
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) c = 0;
    *count = c;
    return SKNNR_OK;
}

int sknnr_host_chunk_plan(int64_t n_q, int64_t chunk_rows, int64_t *rows_out, int32_t cap, int32_t *n_chunks) {
    if (n_q < 0 || chunk_rows < 256 || !n_chunks || (cap > 0 && !rows_out)) return fail(SKNNR_EINVAL, "bad chunk plan arguments");
    const int64_t chunk = std::min<int64_t>((chunk_rows + 255) / 256 * 256, (n_q + 255) / 256 * 256);
    const bool ramp = ramp_applies(false, n_q, chunk);
    int ci = 0;
    for (int64_t r0 = 0, rows = 0; r0 < n_q; r0 += rows, ++ci) {
        rows = next_chunk_rows(ci, n_q - r0, chunk, ramp);
        if (ci < cap) rows_out[ci] = rows;
    }
    *n_chunks = ci;
    return SKNNR_OK;
}

int sknnr_set_option(const char *name, int64_t value) {
    if (!name) return fail(SKNNR_EINVAL, "name is NULL");
    if (!strcmp(name, "engine")) {
        if (value < 0 || value > 3) return fail(SKNNR_EINVAL, "engine must be 0..3");
        g_opt.engine = value;
    } else if (!strcmp(name, "chunk_rows")) {
        if (value < 256) return fail(SKNNR_EINVAL, "chunk_rows must be >= 256");
        g_opt.chunk_rows = (value + 255) / 256 * 256;
    } else if (!strcmp(name, "timing")) {
        g_opt.timing = value ? 1 : 0;
    } else if (!strcmp(name, "kc")) {
        if (value != 0 && value != 8 && value != 16 && value != 32)
            return fail(SKNNR_EINVAL, "kc must be 0, 8, 16 or 32");
        g_opt.kc = value;
    } else if (!strcmp(name, "tc_debug")) {
        g_tc_debug = (int)value;
    } else if (!strcmp(name, "tc_streams")) {
        if (value < 0 || value > 2) return fail(SKNNR_EINVAL, "tc_streams must be 0, 1 or 2");
        g_opt.tc_streams = value;
    } else if (!strcmp(name, "host_slots")) {
        if (value < 1 || value > IndexBase::kSlots) return fail(SKNNR_EINVAL, "host_slots must be 1..8");
        g_opt.host_slots = value;
    } else if (!strcmp(name, "stage_rows")) {
        if (value < 1024) return fail(SKNNR_EINVAL, "stage_rows must be >= 1024");
        g_opt.stage_rows = (value + 1023) / 1024 * 1024;
    } else if (!strcmp(name, "tc_seed_stride")) {
        if (value < 0 || value > 64) return fail(SKNNR_EINVAL, "tc_seed_stride must be 0..64");
        g_opt.tc_seed_stride = value;
    } else {
        return fail(SKNNR_EINVAL, std::string("unknown option ") + name);
    }
    return SKNNR_OK;
}

int sknnr_host_alloc(void **ptr, int64_t bytes) {
    if (!ptr || bytes <= 0) return fail(SKNNR_EINVAL, "bad arguments");
    CK(cudaHostAlloc(ptr, (size_t)bytes, cudaHostAllocDefault));
    return SKNNR_OK;
}
int sknnr_host_free(void *ptr) {
    if (ptr) CK(cudaFreeHost(ptr));
    return SKNNR_OK;
}

// ---- device buffers a multi-process caller shares over NVLink ---------------------------------
int sknnr_device_alloc(int32_t device, void **ptr, int64_t bytes) {
    if (!ptr || bytes <= 0) return fail(SKNNR_EINVAL, "bad arguments");
    CK(cudaSetDevice(device));
    CK(cudaMalloc(ptr, (size_t)bytes));
    return SKNNR_OK;
}
int sknnr_device_free(int32_t device, void *ptr) {
    CK(cudaSetDevice(device));
    if (ptr) CK(cudaFree(ptr));
    return SKNNR_OK;
}
int sknnr_ipc_export(int32_t device, void *ptr, void *handle64) {
    if (!ptr || !handle64) return fail(SKNNR_EINVAL, "NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size is part of the ABI");
    CK(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, ptr));
    memcpy(handle64, &h, 64);
    return SKNNR_OK;
}
int sknnr_ipc_open(int32_t device, const void *handle64, void **ptr) {
    if (!ptr || !handle64) return fail(SKNNR_EINVAL, "NULL argument");
    CK(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    CK(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return SKNNR_OK;
}
int sknnr_ipc_close(int32_t device, void *ptr) {
    CK(cudaSetDevice(device));
    if (ptr) CK(cudaIpcCloseMemHandle(ptr));
    return SKNNR_OK;
}
int sknnr_device_copy(int32_t device, void *dst, const void *src, int64_t bytes, int32_t kind, void *stream) {
    if (!dst || !src || bytes < 0) return fail(SKNNR_EINVAL, "bad arguments");
    CK(cudaSetDevice(device));
    const cudaMemcpyKind kd = kind == 1 ? cudaMemcpyHostToDevice : kind == 2 ? cudaMemcpyDeviceToHost
                                                                             : cudaMemcpyDeviceToDevice;
    CK(cudaMemcpyAsync(dst, src, (size_t)bytes, kd, (cudaStream_t)stream));
    if (kind != 0 || !stream) CK(cudaStreamSynchronize((cudaStream_t)stream));
    return SKNNR_OK;
}

// -----------------------------------------------------------------------------------------
// |x - mu| (Manhattan, Chebyshev) below this bound for the query and every plot: no score of the FP32
// filter (twice the distance, plus rounding) can overflow, so every reference outside a candidate list
// has a finite score and a list that is not full holds every reference
constexpr double kLpNormLimit = 0x1p124;

int sknnr_index_create(const double *fit_z, int64_t n_ref, int32_t d_out, const double *center,
                       const double *scale, const double *proj, int32_t d_in, const double *y,
                       int32_t n_out, int32_t device, sknnr_index **out) {
    return sknnr_index_create_metric(fit_z, n_ref, d_out, center, scale, proj, d_in, y, n_out,
                                     SKNNR_METRIC_EUCLIDEAN, device, out);
}

int sknnr_index_create_metric(const double *fit_z, int64_t n_ref, int32_t d_out, const double *center,
                              const double *scale, const double *proj, int32_t d_in, const double *y,
                              int32_t n_out, int32_t metric, int32_t device, sknnr_index **out) {
    if (!fit_z || !out || n_ref < 1 || d_out < 1 || d_in < 1)
        return fail(SKNNR_EINVAL, "bad arguments to sknnr_index_create");
    if (metric != SKNNR_METRIC_EUCLIDEAN && metric != SKNNR_METRIC_MANHATTAN && metric != SKNNR_METRIC_CHEBYSHEV)
        return fail(SKNNR_EINVAL, "unknown metric");
    if (!proj && d_in != d_out) return fail(SKNNR_EINVAL, "d_in != d_out without a projector");
    if (n_ref >= (1LL << 31) - 64) return fail(SKNNR_EUNSUP, "n_ref too large");
    if (y == nullptr) n_out = 0;
    sknnr_index *ix = new sknnr_index();
    int rc = ix->init_common(device, y, n_ref, n_out);
    if (rc != SKNNR_OK) {
        ix->release_common();
        delete ix;
        return rc;
    }
    ix->metric = metric;
    ix->d_in = d_in;
    ix->d_out = d_out;
    ix->dpad = round_up(d_out, 8);
    ix->n_rtiles = (int)((n_ref + RTILE - 1) / RTILE);

    // centroid of the reference plots: the search images hold (z - mu) so FP32 keeps its
    // precision on raw, uncentred features (UTM-like coordinates)
    std::vector<double> mu(d_out, 0.0);
    for (int64_t j = 0; j < n_ref; ++j)
        for (int k = 0; k < d_out; ++k) mu[k] += fit_z[j * d_out + k];
    for (int k = 0; k < d_out; ++k) mu[k] /= (double)n_ref;

    // reference tile images [(dpad+1)][64] f32, last row = |r|^2 (+inf for padding plots).
    // Manhattan / Chebyshev: -2 (r - mu), the query image's own transform, and a last row of 0 (+inf
    // for padding plots) that starts the sum / maximum.
    const bool lp = metric != SKNNR_METRIC_EUCLIDEAN;
    const size_t tile_floats = (size_t)(ix->dpad + 1) * RTILE;
    std::vector<float> rimg((size_t)ix->n_rtiles * tile_floats, 0.0f);
    double r2max = 0.0;
    for (int t = 0; t < ix->n_rtiles; ++t) {
        float *img = rimg.data() + (size_t)t * tile_floats;
        for (int jj = 0; jj < RTILE; ++jj) {
            const int64_t j = (int64_t)t * RTILE + jj;
            if (j >= n_ref) {
                img[(size_t)ix->dpad * RTILE + jj] = INFINITY;
                continue;
            }
            double n32 = 0.0, n64 = 0.0;
            for (int k = 0; k < d_out; ++k) {
                const double v = fit_z[j * d_out + k] - mu[k];
                if (lp) {
                    img[(size_t)k * RTILE + jj] = (float)(-2.0 * v);
                    n64 = metric == SKNNR_METRIC_MANHATTAN ? n64 + std::fabs(v) : std::max(n64, std::fabs(v));
                    continue;
                }
                const float f = (float)v;
                img[(size_t)k * RTILE + jj] = f;
                n32 += (double)f * (double)f;
                n64 += v * v;
            }
            img[(size_t)ix->dpad * RTILE + jj] = (float)n32;
            r2max = std::max(r2max, n64);
        }
    }
    ix->r2max = r2max;
    if (lp) ix->simt_ok = r2max < kLpNormLimit;   // (false for NaN as well)

    auto up = [&](double **dst, const double *src, size_t n) -> cudaError_t {
        cudaError_t e = cudaMalloc(dst, n * sizeof(double));
        if (e != cudaSuccess) return e;
        return cudaMemcpy(*dst, src, n * sizeof(double), cudaMemcpyHostToDevice);
    };
    cudaError_t e = up(&ix->d_ref64, fit_z, (size_t)n_ref * d_out);
    if (e == cudaSuccess) e = up(&ix->d_mu, mu.data(), d_out);
    if (e == cudaSuccess && center) e = up(&ix->d_center, center, d_in);
    if (e == cudaSuccess && scale) e = up(&ix->d_scale, scale, d_in);
    if (e == cudaSuccess && proj) e = up(&ix->d_proj, proj, (size_t)d_in * d_out);
    if (e == cudaSuccess) e = cudaMalloc(&ix->d_rimg, rimg.size() * sizeof(float));
    if (e == cudaSuccess)
        e = cudaMemcpy(ix->d_rimg, rimg.data(), rimg.size() * sizeof(float), cudaMemcpyHostToDevice);

    // tensor-core engine image: tiles of 128 plots, [chunk][row][8] FP16 (round to nearest even) of
    // sigma * (r - mu), K = d' + 3 padded to a multiple of 16: elements d' .. d'+2 hold a 3-way FP16
    // split of sigma^2 |r - mu|^2 (+inf for padding plots), the rest is zero.  sigma = 2^e scales the
    // plots so that sigma^2 max|r - mu|^2 lies in (2^12, 2^14]: FP16 then keeps its 11-bit significand
    // (the precision of TF32) for every element above 2^-21 of the largest norm, and elements below
    // that (FP16 subnormals, absolute error 2^-25) cannot matter at the certificate's 2^-10.
    const int k_tot = round_up(d_out + 3, 16);
    ix->kc_tot = k_tot / 8;
    ix->n_rtiles_tc = (int)((n_ref + TC_N - 1) / TC_N);
    ix->tc_nstage = search_tc_pick_config(ix->kc_tot);
    // (below a thousand plots a tile pass is a handful of jobs: the FP32 engine is the better filter)
    ix->tensor_ok = !lp && ix->tc_nstage != 0 && std::isfinite(r2max) && n_ref >= 1024;
    if (e == cudaSuccess && ix->tensor_ok) {
        int ex = 0;
        if (r2max > 0.0) {
            int fe;
            std::frexp(16384.0 / r2max, &fe);          // 16384 / r2max = m * 2^fe, m in [0.5, 1)
            ex = (fe - 1) >= 0 ? (fe - 1) / 2 : -((1 - (fe - 1)) / 2);   // floor((fe - 1) / 2)
        }
        ex = std::max(-500, std::min(500, ex));
        ix->tc_sigma = std::ldexp(1.0, ex);
        const double sg = ix->tc_sigma;
        auto f16 = [](double x) -> double { return (double)__half2float(__float2half_rn((float)x)); };
        const size_t op_halves = (size_t)ix->kc_tot * TC_N * 8;
        std::vector<__half> timg((size_t)ix->n_rtiles_tc * op_halves, __float2half_rn(0.0f));
        for (int t = 0; t < ix->n_rtiles_tc; ++t) {
            __half *img = timg.data() + (size_t)t * op_halves;
            auto at = [&](int k, int jj) -> __half & { return img[((size_t)(k / 8) * TC_N + jj) * 8 + (k % 8)]; };
            for (int jj = 0; jj < TC_N; ++jj) {
                const int64_t j = (int64_t)t * TC_N + jj;
                if (j >= n_ref) {
                    at(d_out, jj) = __float2half_rn(INFINITY);
                    continue;
                }
                double n16 = 0.0;
                for (int k = 0; k < d_out; ++k) {
                    const double f = f16((fit_z[j * d_out + k] - mu[k]) * sg);
                    at(k, jj) = __float2half_rn((float)f);
                    n16 += f * f;
                }
                const double hi = f16(n16), mid = f16(n16 - hi), lo = f16(n16 - hi - mid);
                at(d_out, jj) = __float2half_rn((float)hi);
                at(d_out + 1, jj) = __float2half_rn((float)mid);
                at(d_out + 2, jj) = __float2half_rn((float)lo);
            }
        }
        e = cudaMalloc(&ix->d_rimg_tc, timg.size() * sizeof(__half));
        if (e == cudaSuccess)
            e = cudaMemcpy(ix->d_rimg_tc, timg.data(), timg.size() * sizeof(__half), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) {
        sknnr_index_destroy(ix);
        CK(e);
    }
    *out = ix;
    return SKNNR_OK;
}

int sknnr_index_destroy(sknnr_index *ix) {
    if (!ix) return SKNNR_OK;
    ix->release_common();
    cudaFree(ix->d_ref64); cudaFree(ix->d_center); cudaFree(ix->d_scale); cudaFree(ix->d_proj);
    cudaFree(ix->d_mu); cudaFree(ix->d_rimg); cudaFree(ix->d_rimg_tc);
    delete ix;
    return SKNNR_OK;
}

int sknnr_index_stats(sknnr_index *ix, sknnr_stats *out) {
    if (!ix || !out) return fail(SKNNR_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> g(ix->lock);
    cudaSetDevice(ix->device);
    for (auto &s : ix->slots) ix->harvest(s);
    *out = ix->stats;
    return SKNNR_OK;
}

int sknnr_index_cascade_counts(sknnr_index *ix, int64_t *out3) {
    if (!ix || !out3) return fail(SKNNR_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> g(ix->lock);
    cudaSetDevice(ix->device);
    for (auto &s : ix->slots) ix->harvest(s);
    out3[0] = ix->stats.n_fallback;
    out3[1] = ix->n_simt_rows;
    out3[2] = ix->n_exact_rows;
    return SKNNR_OK;
}

// one chunk of a Euclidean-space query, everything enqueued on s.stream.
//
// Engine cascade (every stage is a filter whose result the float64 refine kernel certifies):
//   1. tensor (tcgen05, FP16 operands, eps 2^-10)      -> refine -> uncertified rows list L1
//   1b. tensor again on the compacted rows of L1, each row from the threshold its first pass proved
//       sufficient (no seeding, nothing dropped)       -> refine -> L1b
//   2. SIMT   (FP32 FFMA2 scores, eps ~(2d+8) 2^-24) on the compacted rows of L1b -> refine -> L2
//   3. exact  (float64, exhaustive) on L2
// With engine = SIMT stage 1 is skipped (L1 = all rows); with engine = EXACT only stage 3 runs.
static int run_chunk(sknnr_index *ix, Slot &s, const void *dX, int x_f32, int64_t ldx, bool transformed,
                     int64_t rows, int64_t row0, int k, uint32_t flags, int decimals, int weights,
                     double *o_dist, long long *o_idx, double *o_pred, bool check_finite = false) {
    const bool excl = flags & SKNNR_EXCLUDE_SELF;
    const int kk = k + (excl ? 1 : 0);
    cudaStream_t st = s.stream;
    const int64_t prow = padded_rows(rows);
    if (check_finite) CK(cudaMemsetAsync(s.nonfinite.p, 0, sizeof(int), st));

    int kc = pick_kc(kk, 1);   // 0: k (+1) is beyond the filtered engines' candidate lists -> exhaustive kernel
    if (kc != 0 && g_opt.kc > kc) kc = (int)g_opt.kc;
    const bool lp = ix->metric != SKNNR_METRIC_EUCLIDEAN;   // Manhattan / Chebyshev: SIMT -> refine_lp -> exact
    const bool simt_ok = kc != 0 && search_simt_pick_stages(ix->dpad, kc) != 0 && ix->simt_ok;
    const int ns_layout = g_opt.tc_streams == 1 ? 1 : (kk <= 7 ? 2 : 1);
    ix->ns_in_use = ns_layout;
    const bool tensor_ok = ix->tensor_ok && !ix->tensor_demoted[ns_layout] && kc != 0 && kc <= 16 && simt_ok;
    int engine = (int)g_opt.engine;
    if (engine == SKNNR_ENGINE_AUTO) engine = tensor_ok ? SKNNR_ENGINE_TENSOR : SKNNR_ENGINE_SIMT;
    if (engine == SKNNR_ENGINE_TENSOR && !(ix->tensor_ok && kc != 0 && kc <= 16 && simt_ok))
        engine = SKNNR_ENGINE_SIMT;
    if (engine == SKNNR_ENGINE_SIMT && !simt_ok) engine = SKNNR_ENGINE_EXACT;
    ix->stats.engine = engine;

    FinishParams fp{};
    fp.k = k;
    fp.exclude_self = excl ? 1 : 0;
    fp.deterministic = (flags & SKNNR_DETERMINISTIC) ? 1 : 0;
    fp.round_scale = std::pow(10.0, (double)decimals);
    fp.row_offset = row0;
    fp.out_dist = o_dist;
    fp.out_idx = o_idx;
    fp.weights = weights;
    fp.y = ix->d_y;
    fp.n_ref = (int)ix->n_ref;
    fp.row_map = nullptr;
    fp.n_out = ix->n_out;
    fp.out_pred = o_pred;

    const bool use_tc = engine == SKNNR_ENGINE_TENSOR;
    const bool use_simt_first = engine == SKNNR_ENGINE_SIMT;
    CK(s.z64.reserve((size_t)rows * ix->d_out));
    if (engine != SKNNR_ENGINE_EXACT) CK(s.qimg.reserve((size_t)prow * ix->dpad));
    if (use_tc) CK(s.qimg_tc.reserve((size_t)prow * ix->kc_tot * 8));
    CK(launch_project(dX, x_f32, ldx, rows, transformed ? ix->d_out : ix->d_in, ix->d_out, ix->dpad,
                      transformed ? nullptr : ix->d_center, transformed ? nullptr : ix->d_scale,
                      transformed ? nullptr : ix->d_proj, ix->d_mu, s.z64.p,
                      use_simt_first ? s.qimg.p : nullptr, use_tc ? s.qimg_tc.p : nullptr, ix->kc_tot,
                      ix->tc_sigma, nullptr, check_finite ? s.nonfinite.p : nullptr, st));
    ix->stats.kernel_launches++;
    if (check_finite) {
        CK(cudaMemcpyAsync(&s.h_fb[2], s.nonfinite.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        s.flag_pending = true;
    }

    ExactArgs ea{};
    ea.metric = ix->metric == SKNNR_METRIC_MANHATTAN ? 2 : ix->metric == SKNNR_METRIC_CHEBYSHEV ? 3 : 0;
    ea.z64 = s.z64.p;
    ea.ref64 = ix->d_ref64;
    ea.d = ix->d_out;
    ea.n_q = rows;
    ea.n_ref = (int)ix->n_ref;
    ea.grid = ix->exact_ctas(rows);

    if (engine == SKNNR_ENGINE_EXACT) {
        ea.list = nullptr;
        ea.count = nullptr;
        if (g_opt.timing) CK(s.mark(st));
        CK(ix->launch_exact_chained(ea, fp, kk, st));
        if (g_opt.timing) CK(s.mark(st));
        ix->stats.kernel_launches++;
        return SKNNR_OK;
    }

    CK(s.cand_idx.reserve((size_t)rows * std::max(kc, 16)));
    CK(s.cand_thr.reserve((size_t)rows * 2));
    CK(s.fb.reserve((size_t)rows + 1));
    CK(s.fb2.reserve((size_t)rows + 1));
    CK(cudaMemsetAsync(s.fb.p, 0, sizeof(int), st));
    CK(cudaMemsetAsync(s.fb2.p, 0, sizeof(int), st));

    RefineArgs ra{};
    ra.ref64 = ix->d_ref64;
    ra.mu = ix->d_mu;
    ra.cand_idx = s.cand_idx.p;
    ra.cand_thr = s.cand_thr.p;
    ra.kc = kc;
    ra.d = ix->d_out;
    ra.n_ref = (int)ix->n_ref;
    ra.r2max = ix->r2max;
    // |approx score - true score| <= eps_s * (|q|^2 + max|r|^2)   (DESIGN.md, "certificate")
    //   SIMT  : FP32 rounding of both operands and of |r|^2, plus dpad sequential FP32 FMAs
    //   tensor: FP16 (round-to-nearest, 2^-11 relative; subnormals 2^-25 absolute, < 2^-24 of the
    //           bound's scale - see sknnr_index_create) operands, exact products, FP32 accumulation
    const double eps_simt = (2.0 * ix->dpad + 8.0) * std::ldexp(1.0, -24) * 1.01;
    const double eps_tc = std::ldexp(1.0, -10) * 1.02 + (8.0 * ix->kc_tot) * std::ldexp(1.0, -20) +
                          std::ldexp(1.0, -24);
    ra.thr_scale = 1.0;
    ra.qn_limit = INFINITY;

    const int *stage2_count = nullptr;  // null: stage 2 covers every row of the chunk
    const int *stage2_list = nullptr;   // chunk rows of the compacted stage-2 rows
    if (use_tc) {
        if (g_opt.timing) CK(s.mark(st));
        // two candidate streams per query while k (+1) <= 7 (twice the scanner warps), else one
        int ns = kk <= 7 ? 2 : 1;   // a stream's list keeps at most 7 (ns = 2) / 15 (ns = 1) candidates
        if (g_opt.tc_streams == 1) ns = 1;
        CK(launch_search_tc(s.qimg_tc.p, ix->d_rimg_tc, ix->kc_tot, ix->n_rtiles_tc, rows, ns, ix->tc_nstage,
                            (int)g_opt.tc_seed_stride, ix->tc_wide_joint, s.cand_idx.p,
                            s.cand_thr.p, nullptr, nullptr, st));
        if (g_opt.timing) CK(s.mark(st));
        // (a second pass only pays after the two-stream layout: its joint list holds 11 candidates, the
        // second pass's single stream 15 - the one-stream layout would meet the same 15 again)
        const bool retry = ns == 2;
        if (retry) {
            CK(s.fb_thr.reserve((size_t)rows));
            CK(s.fbm.reserve((size_t)rows + 1));
            CK(cudaMemsetAsync(s.fbm.p, 0, sizeof(int), st));
        }
        ra.kc = 16;
        ra.n_thr = ns;
        ra.z64 = s.z64.p;
        ra.n_q = rows;
        ra.eps_s = eps_tc;
        // the image holds -2 sigma (z - mu) in FP16: every element is finite while 2 sigma |z - mu| < 65504
        ra.thr_scale = 1.0 / (ix->tc_sigma * ix->tc_sigma);
        ra.qn_limit = 0.99 * (32752.0 / ix->tc_sigma) * (32752.0 / ix->tc_sigma);
        ra.fb_count = s.fb.p;
        ra.fb_list = s.fb.p + 1;
        ra.fb_thr = retry ? s.fb_thr.p : nullptr;
        ra.n_rows_dev = nullptr;
        ra.row_map = nullptr;
        CK(launch_refine(ra, fp, st));
        // everything below only concerns the uncertified rows: continue on the slot's tail stream
        CK(cudaEventRecord(s.ev_stage1, st));
        CK(cudaStreamWaitEvent(s.tail_stream, s.ev_stage1, 0));
        st = s.tail_stream;
        CK(s.z64c.reserve((size_t)rows * ix->d_out));
        const int *list = s.fb.p + 1, *count = s.fb.p;
        if (retry) {
            // stage 1b: the same engine once more over the uncertified rows alone, every row starting from
            // the threshold its first pass proved sufficient (retry_threshold): nothing is parked or
            // dropped on the way, the pass costs a few CTAs, and the FP32 engine is left with the rows
            // that have more than 15 references inside the FP16 error margin of their k-th neighbour.
            CK(launch_gather_rows(s.z64.p, ix->d_out, list, count, rows, s.z64c.p, st));
            CK(launch_project(s.z64c.p, 0, ix->d_out, rows, ix->d_out, ix->d_out, ix->dpad, nullptr, nullptr,
                              nullptr, ix->d_mu, nullptr, nullptr, s.qimg_tc.p, ix->kc_tot, ix->tc_sigma, count,
                              nullptr, st));
            // (one stream of 16 whatever the first pass used: what the two-stream layout cannot certify
            // is mostly rows with more references inside the error margin of the k-th neighbour than
            // its joint list of 11 holds)
            CK(launch_search_tc(s.qimg_tc.p, ix->d_rimg_tc, ix->kc_tot, ix->n_rtiles_tc, rows, 1, ix->tc_nstage,
                                (int)g_opt.tc_seed_stride, 0, s.cand_idx.p, s.cand_thr.p, s.fb_thr.p, count, st));
            FinishParams fpb = fp;
            fpb.row_map = list;
            RefineArgs rb = ra;
            rb.z64 = s.z64c.p;
            rb.n_thr = 1;
            rb.fb_count = s.fbm.p;
            rb.fb_list = s.fbm.p + 1;
            rb.fb_thr = nullptr;
            rb.n_rows_dev = count;
            rb.row_map = list;
            CK(launch_refine(rb, fpb, st));
            ix->stats.kernel_launches += 4;
            list = s.fbm.p + 1;
            count = s.fbm.p;
        }
        // stage 2 input: gather the uncertified rows and rebuild their FP32 query image
        CK(launch_gather_rows(s.z64.p, ix->d_out, list, count, rows, s.z64c.p, st));
        CK(launch_project(s.z64c.p, 0, ix->d_out, rows, ix->d_out, ix->d_out, ix->dpad, nullptr, nullptr,
                          nullptr, ix->d_mu, nullptr, s.qimg.p, nullptr, 0, 1.0, count, nullptr, st));
        ix->stats.kernel_launches += 4;
        stage2_count = count;
        stage2_list = list;
    }

    // stage 2 (or the only fast stage): FP32 SIMT engine
    if (g_opt.timing && !use_tc) CK(s.mark(st));
    // (a handful of rows is not worth a scan of the whole reference set by one warp per row block: below
    // kSimtMinRows the stage passes its rows straight on to the exhaustive kernel)
    constexpr int kSimtMinRows = 256;
    const int bypass = stage2_count ? kSimtMinRows : 0;
    CK(launch_search_simt(s.qimg.p, ix->d_rimg, ix->dpad, ix->n_rtiles, rows, kc, s.cand_idx.p,
                          s.cand_thr.p, stage2_count, ix->spread_tail ? ix->n_sm : 0, bypass, st, ix->metric));
    if (g_opt.timing && !use_tc) CK(s.mark(st));
    FinishParams fp2 = fp;
    fp2.row_map = stage2_list;
    ra.kc = kc;
    ra.n_thr = 1;
    ra.z64 = use_tc ? s.z64c.p : s.z64.p;
    ra.n_q = rows;
    ra.eps_s = eps_simt;
    ra.thr_scale = 1.0;
    ra.qn_limit = INFINITY;
    ra.fb_count = s.fb2.p;
    ra.fb_list = s.fb2.p + 1;
    ra.fb_thr = nullptr;
    ra.bypass_rows = bypass;
    ra.n_rows_dev = stage2_count;
    ra.row_map = fp2.row_map;
    if (lp) {
        // |score / 2 - distance| <= eps * (|q - mu| + max_j |r_j - mu|) in the metric's norm (DESIGN.md §2,
        // "Manhattan and Chebyshev"): FP32 rounding of both images and of their difference, plus, for L1, dpad
        // sequential FP32 additions; the 1 % covers the float64 terms (centring, the norms, the distances)
        ra.eps_s = (ix->metric == SKNNR_METRIC_MANHATTAN ? ix->dpad + 2.0 : 2.0) * std::ldexp(1.0, -24) * 1.01;
        ra.thr_scale = 0.5;
        ra.qn_limit = kLpNormLimit;
        // (+ 2^-120: the absolute error of image elements in FP32's subnormal range, at most 2^-150 each,
        // which the relative bound does not cover)
        ra.r2max = ix->r2max + 0x1p-120;
        CK(launch_refine_lp(ra, ix->metric, fp2, st));
        ix->n_simt_rows += rows;   // (the FP32 stage is the first one: every row of the chunk)
    } else {
        CK(launch_refine(ra, fp2, st));
    }
    ix->stats.kernel_launches += 2;

    // stage 3: exhaustive float64 search of whatever is still uncertified (exact ties etc.)
    ea.list = s.fb2.p + 1;
    ea.count = s.fb2.p;
    CK(ix->launch_exact_chained(ea, fp, kk, st));
    ix->stats.kernel_launches++;
    CK(cudaMemcpyAsync(&s.h_fb[0], use_tc ? s.fb.p : s.fb2.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&s.h_fb[1], s.fb2.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    if (stage2_count) CK(cudaMemcpyAsync(&s.h_fb[3], stage2_count, sizeof(int), cudaMemcpyDeviceToHost, st));
    else s.h_fb[3] = 0;
    s.fb_pending = true;
    s.rows_in_flight = use_tc ? rows : 0;
    if (use_tc) {
        CK(cudaEventRecord(s.ev_tail, st));
        s.tail_pending = true;
    }
    return SKNNR_OK;
}

int sknnr_kneighbors(sknnr_index *ix, const void *X, int32_t x_dtype, int64_t n_q, int64_t ldx,
                     int64_t row_offset, int32_t k, uint32_t flags, int32_t decimals,
                     double *out_dist, int64_t *out_idx, int32_t weights, double *out_pred,
                     void *stream) {
    if (!ix) return fail(SKNNR_EINVAL, "index is NULL");
    int kk = 0;
    int rc = check_query_args(ix->n_ref, ix->n_out, n_q, k, flags, weights, X, out_pred, kk);
    if (rc != SKNNR_OK) return rc;
    if (x_dtype != SKNNR_F64 && x_dtype != SKNNR_F32) return fail(SKNNR_EINVAL, "bad x_dtype");
    std::lock_guard<std::mutex> g(ix->lock);
    CK(cudaSetDevice(ix->device));

    const bool excl = flags & SKNNR_EXCLUDE_SELF;
    const bool dev_ptrs = (flags & SKNNR_DEVICE_PTRS) || false;
    bool transformed = flags & SKNNR_TRANSFORMED;
    bool x_on_device = dev_ptrs;
    if (excl) {
        X = ix->d_ref64;
        x_dtype = SKNNR_F64;
        n_q = ix->n_ref;
        ldx = ix->d_out;
        transformed = true;
        x_on_device = true;
    }
    const int cols = transformed ? ix->d_out : ix->d_in;
    if (ldx < cols) return fail(SKNNR_EINVAL, "ldx smaller than the number of features");
    const size_t esz = x_dtype == SKNNR_F32 ? 4 : 8;
    // A synchronous call takes any mix of host and device pointers (unified addressing): device
    // resident X is read in place, and results bound for device memory - this GPU's or a peer's
    // mapped through sknnr_ipc_open - leave each chunk as one copy-engine transfer on the D2H
    // stream, under the kernels of the following chunks.
    if (!dev_ptrs && !x_on_device && is_device_ptr(X)) x_on_device = true;

    cudaStream_t user_stream = dev_ptrs ? (cudaStream_t)stream : nullptr;
    CallGuard guard(ix, user_stream);
    // whatever an earlier call (possibly a device-pointer call on another stream) left running on
    // the slots this call is going to use must be complete before their scratch is reused
    if (dev_ptrs) {
        for (int i = 0; i < 2; ++i) {
            Slot &s = ix->slots[i];
            if (s.last_pending) CK(cudaStreamWaitEvent(user_stream, s.ev_last, 0));
        }
    } else {
        for (auto &s : ix->slots) CK(ix->finish_slot(s));
    }
    for (auto &s : ix->slots) { s.ev_used = 0; s.fb_pending = false; s.flag_pending = false; }
    ix->stats = sknnr_stats{};
    ix->n_simt_rows = ix->n_exact_rows = 0;
    ix->stats.n_queries = n_q;
    ix->saw_nonfinite = false;
    ix->chunk_rows_seen = ix->chunk_fb_seen = ix->chunk_fail_seen = 0;   // the demotion rule looks at this call's chunks only
    if (n_q == 0) { guard.ok = true; return SKNNR_OK; }

    // ordinary NumPy buffers are staged through page-locked slot buffers by the host pool
    const bool stage_in = !x_on_device && is_pageable(X);
    const bool stage_dist = !dev_ptrs && out_dist && is_pageable(out_dist);
    const bool stage_idx = !dev_ptrs && out_idx && is_pageable(out_idx);
    const bool stage_pred = !dev_ptrs && weights != SKNNR_W_NONE && is_pageable(out_pred);
    const bool staged = stage_in || stage_dist || stage_idx || stage_pred;
    const bool check_finite = (flags & SKNNR_CHECK_FINITE) && !dev_ptrs && !excl;
    // device-resident queries have no copies to overlap: twice the chunk (fewer launches and cascade
    // tails; measured +1.8 %), while host buffers prefer the shorter pipeline ramp of the smaller one
    int64_t chunk = dev_ptrs ? 2 * g_opt.chunk_rows : (staged ? std::min(g_opt.stage_rows, g_opt.chunk_rows) : g_opt.chunk_rows);
    chunk = std::min<int64_t>(chunk, (n_q + 255) / 256 * 256);
    const int n_slots = dev_ptrs ? 2 : std::min<int>(4, (int)g_opt.host_slots);
    // Host buffers: the first chunk's H2D copy and the last chunk's D2H copy cannot overlap any
    // kernel, so the stream of chunks ramps up (1/4, 1/2, 1, ...) and down (..., 1/2, 1/4).
    const bool ramp = ramp_applies(dev_ptrs, n_q, chunk);
    int ci = 0;
    int64_t rows = 0;
    // SKNNR_B200_TRACE=1: per-chunk timeline of a host-buffer call on stderr (events on the chunk's stream:
    // enqueued / input arrived / results complete / results delivered, ms since the call began)
    static const bool trace_on = getenv("SKNNR_B200_TRACE") != nullptr;
    struct ChunkTrace { int64_t rows; cudaEvent_t e[4]; double host_ms; };
    std::vector<ChunkTrace> trace;
    cudaEvent_t trace_t0 = nullptr;
    const auto host_t0 = std::chrono::steady_clock::now();
    const bool tracing = trace_on && !dev_ptrs;
    if (tracing) {
        CK(cudaEventCreate(&trace_t0));
        CK(cudaEventRecord(trace_t0, ix->slots[0].stream));
    }
    auto trace_mark = [&](int which, cudaStream_t st) -> cudaError_t {
        if (!tracing) return cudaSuccess;
        cudaError_t e = cudaEventCreate(&trace.back().e[which]);
        return e != cudaSuccess ? e : cudaEventRecord(trace.back().e[which], st);
    };
    for (int64_t r0 = 0; r0 < n_q; r0 += rows, ++ci) {
        rows = next_chunk_rows(ci, n_q - r0, chunk, ramp);
        // the slots alternate: the tail of chunk c (on its slot's tail stream) overlaps the first
        // stage of chunk c + 1 (other slot's buffers)
        Slot &s = ix->slots[ci % n_slots];
        if (!dev_ptrs) {
            CK(ix->finish_slot(s));   // previous chunk on this slot is done, its results delivered
            // adaptive engine choice: if the FP16 filter cannot certify > 5 % of the rows
            // (ill-conditioned features: huge norms relative to neighbour distances) the FP32
            // engine is the better first stage for this index
            if (ix->chunk_rows_seen >= 4096 && ix->chunk_fb_seen * 3 > ix->chunk_rows_seen)
                ix->tensor_demoted[ix->ns_in_use] = true;
        }
        // (the chunk's kernels run on the caller's stream / the pipeline's compute stream, lent to the slot)
        StreamLoan loan(s, dev_ptrs ? user_stream : ix->host_compute, true);
        if (dev_ptrs && s.tail_pending) {   // the slot's buffers are free once its previous tail is done
            CK(cudaStreamWaitEvent(user_stream, s.ev_tail, 0));
            s.tail_pending = false;
        }
        const cudaStream_t cin = ix->h2d_stream, cout = ix->d2h_stream;
        const void *dX;
        int64_t dld = ldx;
        if (tracing) {
            trace.push_back({rows, {nullptr, nullptr, nullptr, nullptr},
                             std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count()});
            CK(trace_mark(0, cin));
        }
        if (x_on_device) {
            dX = (const unsigned char *)X + (size_t)r0 * ldx * esz;
        } else {
            CK(s.x.reserve((size_t)rows * cols * esz));
            const unsigned char *src = (const unsigned char *)X + (size_t)r0 * ldx * esz;
            if (stage_in) {
                CK(s.h_x.reserve((size_t)rows * cols * esz));
                parallel_copy_rows(s.h_x.p, (size_t)cols * esz, src, (size_t)ldx * esz, (size_t)cols * esz, rows);
                CK(cudaMemcpyAsync(s.x.p, s.h_x.p, (size_t)rows * cols * esz, cudaMemcpyDefault, cin));
            } else if (ldx == cols) {
                CK(cudaMemcpyAsync(s.x.p, src, (size_t)rows * cols * esz, cudaMemcpyDefault, cin));
            } else {
                CK(cudaMemcpy2DAsync(s.x.p, (size_t)cols * esz, src, (size_t)ldx * esz, (size_t)cols * esz,
                                     (size_t)rows, cudaMemcpyDefault, cin));
            }
            CK(cudaEventRecord(s.ev_in, cin));
            CK(cudaStreamWaitEvent(s.stream, s.ev_in, 0));
            ix->stats.h2d_bytes += rows * cols * (int64_t)esz;
            dX = s.x.p;
            dld = cols;
        }
        double *o_dist = nullptr, *o_pred = nullptr;
        long long *o_idx = nullptr;
        if (dev_ptrs) {
            if (out_dist) o_dist = out_dist + r0 * k;
            if (out_idx) o_idx = (long long *)out_idx + r0 * k;
            if (weights != SKNNR_W_NONE) o_pred = out_pred + r0 * ix->n_out;
        } else {
            if (out_dist) { CK(s.o_dist.reserve((size_t)rows * k)); o_dist = s.o_dist.p; }
            if (out_idx) { CK(s.o_idx.reserve((size_t)rows * k)); o_idx = s.o_idx.p; }
            if (weights != SKNNR_W_NONE) { CK(s.o_pred.reserve((size_t)rows * ix->n_out)); o_pred = s.o_pred.p; }
        }
        // the last chunk's second stage has nothing to hide under: it is dealt out over all SMs; the
        // others keep to a few SMs, which costs the following chunk's tensor kernel less
        ix->spread_tail = r0 + rows >= n_q;
        CK(trace_mark(1, cin));
        rc = run_chunk(ix, s, dX, x_dtype == SKNNR_F32, dld, transformed, rows, row_offset + r0, k,
                       flags, decimals, weights, o_dist, o_idx, o_pred, check_finite);
        if (rc != SKNNR_OK) return rc;
        if (!dev_ptrs) {
            // the D2H stream picks the results up behind the first stage and the slot's tail
            CK(cudaEventRecord(s.ev_out, s.stream));
            CK(cudaStreamWaitEvent(cout, s.ev_out, 0));
            if (s.tail_pending) CK(cudaStreamWaitEvent(cout, s.ev_tail, 0));  // results complete
            CK(trace_mark(2, cout));
            // D2H straight into page-locked caller memory, else into the slot's staging buffer (the
            // pool copies it out when the slot is next visited)
            auto deliver = [&](void *dst, const void *src, size_t bytes, bool stage, PinBuf<unsigned char> &hb) -> cudaError_t {
                void *to = dst;
                if (stage) {
                    cudaError_t e = hb.reserve(bytes);
                    if (e != cudaSuccess) return e;
                    to = hb.p;
                    s.owed.push_back({dst, hb.p, bytes});
                }
                ix->stats.d2h_bytes += (int64_t)bytes;
                return cudaMemcpyAsync(to, src, bytes, cudaMemcpyDefault, cout);
            };
            if (out_dist) CK(deliver(out_dist + r0 * k, o_dist, (size_t)rows * k * 8, stage_dist, s.h_dist));
            if (out_idx) CK(deliver(out_idx + r0 * k, o_idx, (size_t)rows * k * 8, stage_idx, s.h_idx));
            if (o_pred) CK(deliver(out_pred + r0 * ix->n_out, o_pred, (size_t)rows * ix->n_out * 8, stage_pred, s.h_pred));
            CK(trace_mark(3, cout));
            CK(cudaEventRecord(s.ev_last, cout));
        } else {
            CK(cudaEventRecord(s.ev_last, user_stream));
        }
        s.last_pending = true;   // the slot's buffers are free for reuse once ev_last has passed
    }
    if (!dev_ptrs) {
        for (auto &s : ix->slots) CK(ix->finish_slot(s));
        if (tracing) {
            fprintf(stderr, "sknnr trace: %zu chunks, chunk %lld rows, %d slots; ms since call start: enqueued(host) started in_arrived results_done delivered\n",
                    trace.size(), (long long)chunk, n_slots);
            for (size_t i = 0; i < trace.size(); ++i) {
                float t[4] = {0, 0, 0, 0};
                for (int w = 0; w < 4; ++w) {
                    if (trace[i].e[w]) {
                        cudaEventElapsedTime(&t[w], trace_t0, trace[i].e[w]);
                        cudaEventDestroy(trace[i].e[w]);
                    }
                }
                fprintf(stderr, "  chunk %2zu rows %8lld  %7.2f  %7.2f %7.2f %7.2f %7.2f\n", i, (long long)trace[i].rows,
                        trace[i].host_ms, t[0], t[1], t[2], t[3]);
            }
            cudaEventDestroy(trace_t0);
        }
    } else {
        // results are complete on the caller's stream once both tails have joined it
        for (auto &s : ix->slots)
            if (s.tail_pending) {
                CK(cudaStreamWaitEvent(user_stream, s.ev_tail, 0));
                CK(cudaEventRecord(s.ev_last, user_stream));
                s.tail_pending = false;
            }
    }
    guard.ok = true;
    // a device-pointer call is not synchronised: its counters are harvested by the stats query
    if (check_finite && ix->saw_nonfinite)
        return fail(SKNNR_ENONFINITE, "Input X contains NaN or infinity.");
    return SKNNR_OK;
}

}  // extern "C" (the raster pipeline below is a template)

// Raster front end (scope row f4).  Per block of pixels, on the block's slot stream:
//   A: H2D of the d band segments -> mask + scan -> count to the host        (issued AHEAD blocks early)
//   B: gather (compaction + transpose) -> `run` (the index's chunk pipeline on the compacted rows)
//      -> scatter to band-major layers -> D2H of the layers
// The count is the only value the host waits for; everything else stays asynchronous.
// run(slot, xc, n_valid, first_row, o_dist, o_idx, o_pred) enqueues the search of one block.
template <class IX, class RUN>
static int raster_impl(IX *ix, int d, const void *bands, int32_t x_dtype, int64_t n_pix, int64_t band_stride,
                       int32_t use_nodata, double nodata, int32_t k, uint32_t flags, int32_t weights,
                       double *out_dist, int64_t *out_idx, double *out_pred, double fill_dist,
                       int64_t fill_idx, double fill_pred, int64_t *n_valid_out, RUN run) {
    if (flags & ~(uint32_t)SKNNR_DETERMINISTIC)
        return fail(SKNNR_EINVAL, "the raster calls accept SKNNR_DETERMINISTIC only");
    int kk = 0;
    int rc = check_query_args(ix->n_ref, ix->n_out, n_pix, k, flags, weights, bands, out_pred, kk);
    if (rc != SKNNR_OK) return rc;
    if (x_dtype != SKNNR_F64 && x_dtype != SKNNR_F32) return fail(SKNNR_EINVAL, "bad x_dtype");
    if (band_stride < n_pix) return fail(SKNNR_EINVAL, "band_stride smaller than the number of pixels");
    std::lock_guard<std::mutex> g(ix->lock);
    CK(cudaSetDevice(ix->device));
    const size_t esz = x_dtype == SKNNR_F32 ? 4 : 8;
    CallGuard guard(ix, nullptr);
    for (auto &s : ix->slots) CK(ix->finish_slot(s));
    for (auto &s : ix->slots) { s.ev_used = 0; s.fb_pending = false; s.flag_pending = false; }
    ix->stats = sknnr_stats{};
    ix->n_simt_rows = ix->n_exact_rows = 0;
    ix->chunk_rows_seen = ix->chunk_fb_seen = ix->chunk_fail_seen = 0;
    if (n_valid_out) *n_valid_out = 0;
    if (n_pix == 0) { guard.ok = true; return SKNNR_OK; }

    const int64_t chunk = std::min<int64_t>(g_opt.chunk_rows, (n_pix + 1023) / 1024 * 1024);
    const int64_t n_blocks = (n_pix + chunk - 1) / chunk;
    constexpr int AHEAD = 3;   // < kSlots: a slot is reused only after its previous block's D2H
    auto stage_a = [&](int64_t b) -> int {
        Slot &s = ix->slots[b % IndexBase::kSlots];
        const int64_t p0 = b * chunk, rows = std::min(chunk, n_pix - p0);
        CK(ix->finish_slot(s));   // the slot's previous block is complete
        CK(s.x.reserve((size_t)rows * d * esz));
        CK(s.r_pos.reserve((size_t)rows));
        CK(s.r_cnt.reserve((size_t)(rows + RASTER_GROUP - 1) / RASTER_GROUP + 2));
        CK(cudaMemcpy2DAsync(s.x.p, (size_t)rows * esz, (const unsigned char *)bands + (size_t)p0 * esz,
                             (size_t)band_stride * esz, (size_t)rows * esz, (size_t)d,
                             cudaMemcpyHostToDevice, s.stream));
        ix->stats.h2d_bytes += rows * d * (int64_t)esz;
        const int groups = (int)((rows + RASTER_GROUP - 1) / RASTER_GROUP);
        CK(launch_raster_mask(s.x.p, x_dtype == SKNNR_F32, rows, d, use_nodata, nodata, s.r_pos.p,
                              s.r_cnt.p, s.r_cnt.p + groups + 1, s.stream));
        CK(cudaMemcpyAsync(s.h_cnt, s.r_cnt.p + groups + 1, sizeof(int), cudaMemcpyDeviceToHost, s.stream));
        CK(cudaEventRecord(s.ev_cnt, s.stream));
        ix->stats.kernel_launches += 2;
        return SKNNR_OK;
    };
    int64_t issued = 0, valid_before = 0;
    for (int64_t b = 0; b < n_blocks; ++b) {
        while (issued < n_blocks && issued < b + AHEAD) {
            rc = stage_a(issued++);
            if (rc != SKNNR_OK) return rc;
        }
        Slot &s = ix->slots[b % IndexBase::kSlots];
        const int64_t p0 = b * chunk, rows = std::min(chunk, n_pix - p0);
        CK(cudaEventSynchronize(s.ev_cnt));
        const int64_t nv = *s.h_cnt;
        double *o_dist = nullptr, *o_pred = nullptr;
        long long *o_idx = nullptr;
        // (with nv == 0 the gather only turns the all-zero flags into "-1 = masked")
        CK(s.xc.reserve((size_t)std::max<int64_t>(nv, 1) * d * esz));
        CK(launch_raster_gather(s.x.p, x_dtype == SKNNR_F32, rows, d, s.r_cnt.p, s.r_pos.p, s.xc.p, s.stream));
        ix->stats.kernel_launches++;
        if (nv > 0) {
            if (out_dist) { CK(s.o_dist.reserve((size_t)nv * k)); o_dist = s.o_dist.p; }
            if (out_idx) { CK(s.o_idx.reserve((size_t)nv * k)); o_idx = s.o_idx.p; }
            if (weights != SKNNR_W_NONE) { CK(s.o_pred.reserve((size_t)nv * ix->n_out)); o_pred = s.o_pred.p; }
            rc = run(s, (const void *)s.xc.p, nv, valid_before, o_dist, o_idx, o_pred);
            if (rc != SKNNR_OK) return rc;
            if (s.tail_pending) CK(cudaStreamWaitEvent(s.stream, s.ev_tail, 0));
        }
        ix->stats.n_queries += nv;
        valid_before += nv;
        if (out_dist) {
            CK(s.r_dist.reserve((size_t)rows * k));
            CK(launch_raster_scatter_f64(s.r_pos.p, rows, o_dist, k, fill_dist, s.r_dist.p, rows, s.stream));
            CK(cudaMemcpy2DAsync(out_dist + p0, (size_t)n_pix * 8, s.r_dist.p, (size_t)rows * 8, (size_t)rows * 8,
                                 (size_t)k, cudaMemcpyDeviceToHost, s.stream));
            ix->stats.d2h_bytes += rows * k * 8;
            ix->stats.kernel_launches++;
        }
        if (out_idx) {
            CK(s.r_idx.reserve((size_t)rows * k));
            CK(launch_raster_scatter_i64(s.r_pos.p, rows, o_idx, k, (long long)fill_idx, s.r_idx.p, rows, s.stream));
            CK(cudaMemcpy2DAsync(out_idx + p0, (size_t)n_pix * 8, s.r_idx.p, (size_t)rows * 8, (size_t)rows * 8,
                                 (size_t)k, cudaMemcpyDeviceToHost, s.stream));
            ix->stats.d2h_bytes += rows * k * 8;
            ix->stats.kernel_launches++;
        }
        if (weights != SKNNR_W_NONE) {
            CK(s.r_pred.reserve((size_t)rows * ix->n_out));
            CK(launch_raster_scatter_f64(s.r_pos.p, rows, o_pred, ix->n_out, fill_pred, s.r_pred.p, rows, s.stream));
            CK(cudaMemcpy2DAsync(out_pred + p0, (size_t)n_pix * 8, s.r_pred.p, (size_t)rows * 8, (size_t)rows * 8,
                                 (size_t)ix->n_out, cudaMemcpyDeviceToHost, s.stream));
            ix->stats.d2h_bytes += rows * ix->n_out * 8;
            ix->stats.kernel_launches++;
        }
    }
    for (auto &s : ix->slots) CK(ix->finish_slot(s));
    guard.ok = true;
    if (n_valid_out) *n_valid_out = valid_before;
    return SKNNR_OK;
}

extern "C" {

int sknnr_raster_kneighbors(sknnr_index *ix, const void *bands, int32_t x_dtype, int64_t n_pix,
                            int64_t band_stride, int32_t use_nodata, double nodata, int32_t k,
                            uint32_t flags, int32_t decimals, double *out_dist, int64_t *out_idx,
                            int32_t weights, double *out_pred, double fill_dist, int64_t fill_idx,
                            double fill_pred, int64_t *n_valid_out) {
    if (!ix) return fail(SKNNR_EINVAL, "index is NULL");
    return raster_impl(ix, ix->d_in, bands, x_dtype, n_pix, band_stride, use_nodata, nodata, k, flags, weights,
                       out_dist, out_idx, out_pred, fill_dist, fill_idx, fill_pred, n_valid_out,
                       [&](Slot &s, const void *xc, int64_t nv, int64_t row0, double *o_dist, long long *o_idx,
                           double *o_pred) -> int {
                           if (ix->chunk_rows_seen >= 4096 && ix->chunk_fb_seen * 3 > ix->chunk_rows_seen)
                               ix->tensor_demoted[ix->ns_in_use] = true;
                           ix->spread_tail = false;
                           return run_chunk(ix, s, xc, x_dtype == SKNNR_F32, ix->d_in, false, nv, row0, k, flags,
                                            decimals, weights, o_dist, o_idx, o_pred);
                       });
}

int sknnr_transform(sknnr_index *ix, const void *X, int32_t x_dtype, int64_t n_q, int64_t ldx,
                    double *out_z) {
    if (!ix || !X || !out_z || n_q < 0) return fail(SKNNR_EINVAL, "NULL argument");
    if (ldx < ix->d_in) return fail(SKNNR_EINVAL, "ldx smaller than the number of features");
    std::lock_guard<std::mutex> g(ix->lock);
    CK(cudaSetDevice(ix->device));
    const size_t esz = x_dtype == SKNNR_F32 ? 4 : 8;
    Slot &s = ix->slots[0];
    const int64_t chunk = g_opt.chunk_rows;
    for (int64_t r0 = 0; r0 < n_q; r0 += chunk) {
        const int64_t rows = std::min(chunk, n_q - r0);
        CK(s.x.reserve((size_t)rows * ix->d_in * esz));
        CK(s.z64.reserve((size_t)rows * ix->d_out));
        CK(cudaMemcpy2DAsync(s.x.p, (size_t)ix->d_in * esz, (const unsigned char *)X + (size_t)r0 * ldx * esz,
                             (size_t)ldx * esz, (size_t)ix->d_in * esz, (size_t)rows,
                             cudaMemcpyHostToDevice, s.stream));
        CK(launch_project(s.x.p, x_dtype == SKNNR_F32, ix->d_in, rows, ix->d_in, ix->d_out, ix->dpad,
                          ix->d_center, ix->d_scale, ix->d_proj, ix->d_mu, s.z64.p, nullptr, nullptr, 0, 1.0, nullptr, nullptr,
                          s.stream));
        CK(cudaMemcpyAsync(out_z + r0 * ix->d_out, s.z64.p, (size_t)rows * ix->d_out * 8,
                           cudaMemcpyDeviceToHost, s.stream));
        CK(cudaStreamSynchronize(s.stream));
    }
    return SKNNR_OK;
}

static int weighted_average_common(IndexBase *ix, const int64_t *idx, const double *w, int64_t n_q,
                                   int32_t k, double *out_pred) {
    if (!ix || !idx || !w || !out_pred || n_q < 0 || k < 1) return fail(SKNNR_EINVAL, "NULL argument");
    if (!ix->d_y) return fail(SKNNR_EINVAL, "index was built without targets");
    std::lock_guard<std::mutex> g(ix->lock);
    CK(cudaSetDevice(ix->device));
    Slot &s = ix->slots[0];
    CK(s.o_idx.reserve((size_t)n_q * k));
    CK(s.o_dist.reserve((size_t)n_q * k));
    CK(s.o_pred.reserve((size_t)n_q * ix->n_out));
    CK(cudaMemcpyAsync(s.o_idx.p, idx, (size_t)n_q * k * 8, cudaMemcpyHostToDevice, s.stream));
    CK(cudaMemcpyAsync(s.o_dist.p, w, (size_t)n_q * k * 8, cudaMemcpyHostToDevice, s.stream));
    CK(launch_weighted_average(s.o_idx.p, s.o_dist.p, n_q, k, ix->d_y, ix->n_out, s.o_pred.p, s.stream));
    CK(cudaMemcpyAsync(out_pred, s.o_pred.p, (size_t)n_q * ix->n_out * 8, cudaMemcpyDeviceToHost, s.stream));
    CK(cudaStreamSynchronize(s.stream));
    return SKNNR_OK;
}

int sknnr_weighted_average(sknnr_index *ix, const int64_t *idx, const double *w, int64_t n_q,
                           int32_t k, double *out_pred) {
    return weighted_average_common(ix, idx, w, n_q, k, out_pred);
}

// -----------------------------------------------------------------------------------------
int sknnr_hamming_index_create(const uint16_t *ref_codes, int64_t n_ref, int32_t n_trees,
                               const double *w, const double *y, int32_t n_out, int32_t device,
                               sknnr_hamming_index **out) {
    if (!ref_codes || !w || !out || n_ref < 1 || n_trees < 1)
        return fail(SKNNR_EINVAL, "bad arguments to sknnr_hamming_index_create");
    if (n_ref >= (1LL << 31) - 64) return fail(SKNNR_EUNSUP, "n_ref too large");
    for (int64_t e = 0; e < n_ref * (int64_t)n_trees; ++e)
        if (ref_codes[e] > 31743) return fail(SKNNR_EINVAL, "node codes must be <= 31743");
    if (y == nullptr) n_out = 0;
    sknnr_hamming_index *ix = new sknnr_hamming_index();
    int rc = ix->init_common(device, y, n_ref, n_out);
    if (rc != SKNNR_OK) {
        ix->release_common();
        delete ix;
        return rc;
    }
    ix->n_trees = n_trees;
    ix->n_chunks = (n_trees + 2 * HAM_WC - 1) / (2 * HAM_WC);
    ix->n_rtiles = (int)((n_ref + RTILE - 1) / RTILE);
    ix->uniform = true;
    for (int t = 1; t < n_trees; ++t)
        if (w[t] != w[0]) ix->uniform = false;
    // SciPy's denominators / numerators are left-to-right float64 sums
    volatile double den = 0.0;
    for (int t = 0; t < n_trees; ++t) den = den + w[t];
    ix->wsum = den;
    std::vector<double> lut(n_trees + 1, 0.0);
    volatile double acc = 0.0;
    for (int m = 1; m <= n_trees; ++m) {
        acc = acc + w[0];
        lut[m] = acc / den;
    }
    // Fixed-point weights of the filter: w_t = scale * wq_t + e_t, wq_t in [0, 65535].  The certificate
    // needs sum |e_t| plus the rounding of two left-to-right float64 sums (DESIGN.md, "weighted Hamming").
    std::vector<uint32_t> wq((size_t)ix->n_chunks * HAM_WC, 0u);
    {
        double wmax = 0.0;
        bool okw = true;
        for (int t = 0; t < n_trees; ++t) {
            if (!(w[t] >= 0.0) || !std::isfinite(w[t])) okw = false;
            wmax = std::max(wmax, w[t]);
        }
        ix->wq_ok = okw && wmax > 0.0 && std::isfinite(den) && n_trees <= 32768;
        if (ix->wq_ok) {
            const double scale = wmax / 65535.0;
            double err = 0.0;
            for (int t = 0; t < n_trees; ++t) {
                double qv = std::nearbyint(w[t] / scale);
                qv = std::min(65535.0, std::max(0.0, qv));
                err += std::fabs(w[t] - scale * qv);
                wq[t / 2] |= (uint32_t)qv << (16 * (t & 1));
            }
            ix->wq_scale = scale;
            ix->wq_err = err * (1.0 + 1e-9) + 4.0 * n_trees * std::ldexp(1.0, -53) * den;
        }
    }
    cudaError_t e = cudaMalloc(&ix->d_rcodes, (size_t)n_ref * n_trees * 2);
    if (e == cudaSuccess) e = cudaMalloc(&ix->d_wq, wq.size() * 4);
    if (e == cudaSuccess) e = cudaMemcpy(ix->d_wq, wq.data(), wq.size() * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess)
        e = cudaMemcpy(ix->d_rcodes, ref_codes, (size_t)n_ref * n_trees * 2, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&ix->d_w, (size_t)n_trees * 8);
    if (e == cudaSuccess) e = cudaMemcpy(ix->d_w, w, (size_t)n_trees * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&ix->d_lut, lut.size() * 8);
    if (e == cudaSuccess) e = cudaMemcpy(ix->d_lut, lut.data(), lut.size() * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess)
        e = cudaMalloc(&ix->d_rimg, (size_t)ix->n_rtiles * ix->n_chunks * HAM_WC * RTILE * 4);
    if (e == cudaSuccess)
        e = launch_hamming_pack(ix->d_rcodes, n_ref, n_trees, n_trees, ix->n_chunks, RTILE, 31743,
                                ix->d_rimg, 0);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        sknnr_hamming_index_destroy(ix);
        CK(e);
    }
    *out = ix;
    return SKNNR_OK;
}

int sknnr_hamming_index_destroy(sknnr_hamming_index *ix) {
    if (!ix) return SKNNR_OK;
    ix->release_common();
    cudaFree(ix->d_rcodes); cudaFree(ix->d_rimg); cudaFree(ix->d_w); cudaFree(ix->d_lut);
    cudaFree(ix->d_wq);
    delete ix;
    return SKNNR_OK;
}

int sknnr_hamming_index_stats(sknnr_hamming_index *ix, sknnr_stats *out) {
    if (!ix || !out) return fail(SKNNR_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> g(ix->lock);
    cudaSetDevice(ix->device);
    for (auto &s : ix->slots) ix->harvest(s);
    *out = ix->stats;
    return SKNNR_OK;
}

static int run_hamming_chunk(sknnr_hamming_index *ix, Slot &s, const uint16_t *dq, int64_t ldq,
                             int64_t rows, int64_t row0, int k, uint32_t flags, int decimals,
                             int weights, double *o_dist, long long *o_idx, double *o_pred) {
    const bool excl = flags & SKNNR_EXCLUDE_SELF;
    const int kk = k + (excl ? 1 : 0);
    cudaStream_t st = s.stream;
    FinishParams fp{};
    fp.k = k;
    fp.exclude_self = excl ? 1 : 0;
    fp.deterministic = (flags & SKNNR_DETERMINISTIC) ? 1 : 0;
    fp.round_scale = std::pow(10.0, (double)decimals);
    fp.row_offset = row0;
    fp.out_dist = o_dist;
    fp.out_idx = o_idx;
    fp.weights = weights;
    fp.y = ix->d_y;
    fp.n_ref = (int)ix->n_ref;
    fp.n_out = ix->n_out;
    fp.out_pred = o_pred;

    // equal weights: integer counts are exact, kc = k suffices.  Unequal weights: the fixed-point
    // filter keeps >= 8 spare candidates for the certificate of hamming_refine_kernel.
    const bool exact_only = g_opt.engine == SKNNR_ENGINE_EXACT;
    const int kc_u = pick_kc(kk, 0);
    const int kc_w = std::max(16, pick_kc(kk, 8));
    const bool fast_u = ix->uniform && kc_u != 0 && ix->n_chunks * HAM_WC <= 2048 && !exact_only;
    const bool fast_w = !fast_u && !ix->uniform && ix->wq_ok && pick_kc(kk, 8) != 0 && !exact_only;
    ix->stats.engine = (fast_u || fast_w) ? SKNNR_ENGINE_SIMT : SKNNR_ENGINE_EXACT;

    ExactArgs ea{};
    ea.metric = 1;
    ea.qcodes = dq;
    ea.ldq = ldq;
    ea.rcodes = ix->d_rcodes;
    ea.n_trees = ix->n_trees;
    ea.w = ix->d_w;
    ea.wsum = ix->wsum;
    ea.n_q = rows;
    ea.n_ref = (int)ix->n_ref;
    ea.grid = ix->exact_ctas(rows);
    if (!fast_u && !fast_w) {
        if (g_opt.timing) CK(s.mark(st));
        CK(ix->launch_exact_chained(ea, fp, kk, st));
        if (g_opt.timing) CK(s.mark(st));
        ix->stats.kernel_launches++;
        return SKNNR_OK;
    }
    const int kc = fast_u ? kc_u : kc_w;
    const int64_t n_qtiles = (rows + QTILE - 1) / QTILE;
    CK(s.qimg_h.reserve((size_t)n_qtiles * ix->n_chunks * HAM_WC * QTILE));
    CK(s.cand_idx.reserve((size_t)rows * kc));
    CK(s.cand_cnt.reserve((size_t)rows * kc));
    CK(launch_hamming_pack(dq, rows, ldq, ix->n_trees, ix->n_chunks, QTILE, 31743, s.qimg_h.p, st));
    if (g_opt.timing) CK(s.mark(st));
    CK(launch_hamming_search(s.qimg_h.p, ix->d_rimg, fast_w ? ix->d_wq : nullptr, ix->n_chunks, ix->n_rtiles,
                             rows, (int)ix->n_ref, kc, s.cand_idx.p, s.cand_cnt.p, st));
    if (g_opt.timing) CK(s.mark(st));
    if (fast_u) {
        CK(launch_hamming_finish(s.cand_idx.p, s.cand_cnt.p, kc, ix->d_lut, rows, fp, st));
        ix->stats.kernel_launches += 3;
        return SKNNR_OK;
    }
    CK(s.fb.reserve((size_t)rows + 1));
    CK(cudaMemsetAsync(s.fb.p, 0, sizeof(int), st));
    HammingRefineArgs ha{};
    ha.cand_idx = s.cand_idx.p;
    ha.cand_cnt = s.cand_cnt.p;
    ha.kc = kc;
    ha.qcodes = dq;
    ha.ldq = ldq;
    ha.rcodes = ix->d_rcodes;
    ha.n_trees = ix->n_trees;
    ha.w = ix->d_w;
    ha.wsum = ix->wsum;
    ha.scale = ix->wq_scale;
    ha.err = ix->wq_err;
    ha.n_q = rows;
    ha.fb_count = s.fb.p;
    ha.fb_list = s.fb.p + 1;
    CK(launch_hamming_refine(ha, fp, st));
    // exhaustive float64 search of the uncertified rows
    ea.list = s.fb.p + 1;
    ea.count = s.fb.p;
    CK(ix->launch_exact_chained(ea, fp, kk, st));
    CK(cudaMemcpyAsync(&s.h_fb[0], s.fb.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    s.h_fb[1] = 0;
    s.fb_pending = true;
    s.rows_in_flight = 0;
    ix->stats.kernel_launches += 4;
    return SKNNR_OK;
}

// Shared body of sknnr_hamming_kneighbors (forest == NULL: `q` holds u16 node codes, row stride
// ldq elements) and sknnr_hamming_kneighbors_forest (`q` holds raw feature rows of x_dtype, row
// stride ldq elements; every chunk is walked through the forest on the device first).
static int hamming_kneighbors_impl(sknnr_hamming_index *ix, sknnr_forest *forest, const void *q,
                                   int32_t x_dtype, int64_t n_q, int64_t ldq, int64_t row_offset,
                                   int32_t k, uint32_t flags, int32_t decimals, double *out_dist,
                                   int64_t *out_idx, int32_t weights, double *out_pred, void *stream) {
    if (!ix) return fail(SKNNR_EINVAL, "index is NULL");
    const uint16_t *q_codes = forest ? nullptr : (const uint16_t *)q;
    int kk = 0;
    int rc = check_query_args(ix->n_ref, ix->n_out, n_q, k, flags, weights, q, out_pred, kk);
    if (rc != SKNNR_OK) return rc;
    if (forest) {
        if (forest->n_trees != ix->n_trees) return fail(SKNNR_EINVAL, "forest and index disagree on the number of trees");
        if (forest->device != ix->device) return fail(SKNNR_EINVAL, "forest and index live on different devices");
        if (x_dtype != SKNNR_F64 && x_dtype != SKNNR_F32) return fail(SKNNR_EINVAL, "bad x_dtype");
    }
    std::lock_guard<std::mutex> g(ix->lock);
    CK(cudaSetDevice(ix->device));
    const bool excl = flags & SKNNR_EXCLUDE_SELF;
    const bool dev_ptrs = flags & SKNNR_DEVICE_PTRS;
    bool q_on_device = dev_ptrs;
    if (excl) {
        forest = nullptr;   // X=None: the reference plots' own codes
        q_codes = ix->d_rcodes;
        n_q = ix->n_ref;
        ldq = ix->n_trees;
        q_on_device = true;
    }
    if (!forest && ldq < ix->n_trees) return fail(SKNNR_EINVAL, "ldq smaller than the number of trees");
    if (forest && ldq < forest->n_features) return fail(SKNNR_EINVAL, "ldx smaller than the number of features");
    const size_t xesz = x_dtype == SKNNR_F32 ? 4 : 8;
    cudaStream_t user_stream = dev_ptrs ? (cudaStream_t)stream : nullptr;
    CallGuard guard(ix, user_stream);
    if (dev_ptrs) {
        if (ix->slots[0].last_pending) CK(cudaStreamWaitEvent(user_stream, ix->slots[0].ev_last, 0));
    } else {
        for (auto &s : ix->slots) CK(ix->finish_slot(s));
    }
    for (auto &s : ix->slots) { s.ev_used = 0; s.fb_pending = false; s.flag_pending = false; }
    ix->stats = sknnr_stats{};
    ix->stats.n_queries = n_q;
    if (n_q == 0) { guard.ok = true; return SKNNR_OK; }
    const int64_t chunk = std::min<int64_t>(g_opt.chunk_rows, (n_q + 255) / 256 * 256);
    int ci = 0;
    for (int64_t r0 = 0; r0 < n_q; r0 += chunk, ++ci) {
        const int64_t rows = std::min(chunk, n_q - r0);
        Slot &s = dev_ptrs ? ix->slots[0] : ix->slots[ci % IndexBase::kSlots];
        StreamLoan loan(s, user_stream, dev_ptrs);
        if (!dev_ptrs) CK(ix->finish_slot(s));
        const uint16_t *dq;
        int64_t dld = ldq;
        if (forest) {
            // raw feature rows -> device -> forest walk -> 16-bit node codes, all on s.stream
            const void *dX;
            int64_t dldx = ldq;
            if (q_on_device) {
                dX = (const unsigned char *)q + (size_t)r0 * ldq * xesz;
            } else {
                const int64_t cols = forest->n_features;
                CK(s.x.reserve((size_t)rows * cols * xesz));
                CK(cudaMemcpy2DAsync(s.x.p, (size_t)cols * xesz, (const unsigned char *)q + (size_t)r0 * ldq * xesz,
                                     (size_t)ldq * xesz, (size_t)cols * xesz, (size_t)rows,
                                     cudaMemcpyHostToDevice, s.stream));
                ix->stats.h2d_bytes += rows * cols * (int64_t)xesz;
                dX = s.x.p;
                dldx = cols;
            }
            CK(s.codes.reserve((size_t)rows * ix->n_trees));
            CK(launch_forest_apply(dX, x_dtype == SKNNR_F32, dldx, rows, forest->n_features, forest->d_nodes,
                                   forest->d_roots, forest->n_trees, s.codes.p, nullptr, ix->n_trees, s.stream));
            ix->stats.kernel_launches++;
            dq = s.codes.p;
            dld = ix->n_trees;
        } else if (q_on_device) {
            dq = q_codes + (size_t)r0 * ldq;
        } else {
            CK(s.x.reserve((size_t)rows * ix->n_trees * 2));
            CK(cudaMemcpy2DAsync(s.x.p, (size_t)ix->n_trees * 2, q_codes + (size_t)r0 * ldq,
                                 (size_t)ldq * 2, (size_t)ix->n_trees * 2, (size_t)rows,
                                 cudaMemcpyHostToDevice, s.stream));
            ix->stats.h2d_bytes += rows * ix->n_trees * 2;
            dq = (const uint16_t *)s.x.p;
            dld = ix->n_trees;
        }
        double *o_dist = nullptr, *o_pred = nullptr;
        long long *o_idx = nullptr;
        if (dev_ptrs) {
            if (out_dist) o_dist = out_dist + r0 * k;
            if (out_idx) o_idx = (long long *)out_idx + r0 * k;
            if (weights != SKNNR_W_NONE) o_pred = out_pred + r0 * ix->n_out;
        } else {
            if (out_dist) { CK(s.o_dist.reserve((size_t)rows * k)); o_dist = s.o_dist.p; }
            if (out_idx) { CK(s.o_idx.reserve((size_t)rows * k)); o_idx = s.o_idx.p; }
            if (weights != SKNNR_W_NONE) { CK(s.o_pred.reserve((size_t)rows * ix->n_out)); o_pred = s.o_pred.p; }
        }
        rc = run_hamming_chunk(ix, s, dq, dld, rows, row_offset + r0, k, flags, decimals, weights,
                               o_dist, o_idx, o_pred);
        if (rc != SKNNR_OK) return rc;
        if (!dev_ptrs) {
            if (out_dist) {
                CK(cudaMemcpyAsync(out_dist + r0 * k, o_dist, (size_t)rows * k * 8, cudaMemcpyDeviceToHost, s.stream));
                ix->stats.d2h_bytes += rows * k * 8;
            }
            if (out_idx) {
                CK(cudaMemcpyAsync(out_idx + r0 * k, o_idx, (size_t)rows * k * 8, cudaMemcpyDeviceToHost, s.stream));
                ix->stats.d2h_bytes += rows * k * 8;
            }
            if (o_pred) {
                CK(cudaMemcpyAsync(out_pred + r0 * ix->n_out, o_pred, (size_t)rows * ix->n_out * 8, cudaMemcpyDeviceToHost, s.stream));
                ix->stats.d2h_bytes += rows * ix->n_out * 8;
            }
        } else {
            CK(cudaEventRecord(s.ev_last, user_stream));
            s.last_pending = true;
        }
    }
    if (!dev_ptrs)
        for (auto &s : ix->slots) CK(ix->finish_slot(s));
    guard.ok = true;
    return SKNNR_OK;
}

// Raster front end for the tree-node estimators: band-major pixels -> compacted feature rows ->
// forest walk -> node codes -> Hamming search -> band-major layers, all on the device.
int sknnr_hamming_raster_kneighbors_forest(sknnr_hamming_index *ix, sknnr_forest *forest, const void *bands,
                                           int32_t x_dtype, int64_t n_pix, int64_t band_stride,
                                           int32_t use_nodata, double nodata, int32_t k, uint32_t flags,
                                           int32_t decimals, double *out_dist, int64_t *out_idx,
                                           int32_t weights, double *out_pred, double fill_dist,
                                           int64_t fill_idx, double fill_pred, int64_t *n_valid_out) {
    if (!ix || !forest) return fail(SKNNR_EINVAL, "index or forest is NULL");
    if (forest->n_trees != ix->n_trees) return fail(SKNNR_EINVAL, "forest and index disagree on the number of trees");
    if (forest->device != ix->device) return fail(SKNNR_EINVAL, "forest and index live on different devices");
    return raster_impl(ix, forest->n_features, bands, x_dtype, n_pix, band_stride, use_nodata, nodata, k, flags,
                       weights, out_dist, out_idx, out_pred, fill_dist, fill_idx, fill_pred, n_valid_out,
                       [&](Slot &s, const void *xc, int64_t nv, int64_t row0, double *o_dist, long long *o_idx,
                           double *o_pred) -> int {
                           CK(s.codes.reserve((size_t)nv * ix->n_trees));
                           CK(launch_forest_apply(xc, x_dtype == SKNNR_F32, forest->n_features, nv,
                                                  forest->n_features, forest->d_nodes, forest->d_roots,
                                                  forest->n_trees, s.codes.p, nullptr, ix->n_trees, s.stream));
                           ix->stats.kernel_launches++;
                           return run_hamming_chunk(ix, s, s.codes.p, ix->n_trees, nv, row0, k, flags, decimals,
                                                    weights, o_dist, o_idx, o_pred);
                       });
}

int sknnr_hamming_kneighbors(sknnr_hamming_index *ix, const uint16_t *q_codes, int64_t n_q,
                             int64_t ldq, int64_t row_offset, int32_t k, uint32_t flags,
                             int32_t decimals, double *out_dist, int64_t *out_idx,
                             int32_t weights, double *out_pred, void *stream) {
    return hamming_kneighbors_impl(ix, nullptr, q_codes, 0, n_q, ldq, row_offset, k, flags, decimals,
                                   out_dist, out_idx, weights, out_pred, stream);
}

int sknnr_hamming_kneighbors_forest(sknnr_hamming_index *ix, sknnr_forest *forest, const void *X,
                                    int32_t x_dtype, int64_t n_q, int64_t ldx, int64_t row_offset,
                                    int32_t k, uint32_t flags, int32_t decimals, double *out_dist,
                                    int64_t *out_idx, int32_t weights, double *out_pred, void *stream) {
    if (!forest) return fail(SKNNR_EINVAL, "forest is NULL");
    return hamming_kneighbors_impl(ix, forest, X, x_dtype, n_q, ldx, row_offset, k, flags, decimals,
                                   out_dist, out_idx, weights, out_pred, stream);
}

// -----------------------------------------------------------------------------------------
int sknnr_forest_create(const int32_t *tree_offsets, const int32_t *children_left,
                        const int32_t *children_right, const int32_t *feature, const double *threshold,
                        const uint8_t *missing_go_to_left, const uint16_t *node_code, int32_t n_trees,
                        int32_t n_features, int32_t device, sknnr_forest **out) {
    if (!tree_offsets || !children_left || !children_right || !feature || !threshold || !out || n_trees < 1 ||
        n_features < 1)
        return fail(SKNNR_EINVAL, "bad arguments to sknnr_forest_create");
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
        return fail(SKNNR_ENODEV, "no CUDA device: sknnr_b200 has no CPU fallback");
    if (device < 0 || device >= count) return fail(SKNNR_EINVAL, "bad device ordinal");
    if (forest_smem_bytes(n_features) > 227 * 1024) return fail(SKNNR_EUNSUP, "too many features for the forest kernel");
    const long long n_nodes = tree_offsets[n_trees];
    if (n_nodes < n_trees) return fail(SKNNR_EINVAL, "bad tree offsets");
    std::vector<ForestNode> nodes((size_t)n_nodes);
    std::vector<int> roots(n_trees);
    for (int t = 0; t < n_trees; ++t) {
        const int lo = tree_offsets[t], hi = tree_offsets[t + 1];
        if (hi <= lo) return fail(SKNNR_EINVAL, "empty tree");
        roots[t] = lo;
        for (int i = lo; i < hi; ++i) {
            ForestNode nd{};
            const int l = children_left[i], r = children_right[i];
            if (l < 0) {   // leaf ($SP/sklearn/tree/_tree.pyx: TREE_LEAF = -1)
                nd.left = -1;
                nd.right = node_code ? (int)node_code[i] : (i - lo);   // leaf: the node's code
            } else {
                if (l >= hi - lo || r < 0 || r >= hi - lo) return fail(SKNNR_EINVAL, "child index out of range");
                if (feature[i] < 0 || feature[i] >= n_features) return fail(SKNNR_EINVAL, "feature index out of range");
                nd.left = lo + l;
                nd.right = lo + r;
                // largest float32 <= threshold (exact for float32 feature values, see ForestNode)
                float tf = (float)threshold[i];
                if ((double)tf > threshold[i]) tf = std::nextafterf(tf, -INFINITY);
                nd.thr = tf;
                nd.feat = feature[i] | ((missing_go_to_left && missing_go_to_left[i]) ? (int)0x80000000u : 0);
            }
            nodes[(size_t)i] = nd;
        }
    }
    sknnr_forest *f = new sknnr_forest();
    f->device = device;
    f->n_trees = n_trees;
    f->n_features = n_features;
    f->n_nodes = n_nodes;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaMalloc(&f->d_nodes, nodes.size() * sizeof(ForestNode));
    if (e == cudaSuccess) e = cudaMemcpy(f->d_nodes, nodes.data(), nodes.size() * sizeof(ForestNode), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&f->d_roots, roots.size() * sizeof(int));
    if (e == cudaSuccess) e = cudaMemcpy(f->d_roots, roots.data(), roots.size() * sizeof(int), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&f->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        sknnr_forest_destroy(f);
        CK(e);
    }
    *out = f;
    return SKNNR_OK;
}

int sknnr_forest_destroy(sknnr_forest *f) {
    if (!f) return SKNNR_OK;
    cudaSetDevice(f->device);
    if (f->stream) cudaStreamDestroy(f->stream);
    cudaFree(f->d_nodes);
    cudaFree(f->d_roots);
    f->x.release();
    f->ids.release();
    delete f;
    return SKNNR_OK;
}

int sknnr_forest_apply(sknnr_forest *f, const void *X, int32_t x_dtype, int64_t n_q, int64_t ldx,
                       int32_t *out_ids) {
    if (!f || !X || !out_ids || n_q < 0) return fail(SKNNR_EINVAL, "NULL argument");
    if (ldx < f->n_features) return fail(SKNNR_EINVAL, "ldx smaller than the number of features");
    if (x_dtype != SKNNR_F64 && x_dtype != SKNNR_F32) return fail(SKNNR_EINVAL, "bad x_dtype");
    std::lock_guard<std::mutex> g(f->lock);
    CK(cudaSetDevice(f->device));
    const size_t esz = x_dtype == SKNNR_F32 ? 4 : 8;
    const int64_t chunk = g_opt.chunk_rows;
    for (int64_t r0 = 0; r0 < n_q; r0 += chunk) {
        const int64_t rows = std::min(chunk, n_q - r0);
        CK(f->x.reserve((size_t)rows * f->n_features * esz));
        CK(f->ids.reserve((size_t)rows * f->n_trees));
        CK(cudaMemcpy2DAsync(f->x.p, (size_t)f->n_features * esz, (const unsigned char *)X + (size_t)r0 * ldx * esz,
                             (size_t)ldx * esz, (size_t)f->n_features * esz, (size_t)rows, cudaMemcpyHostToDevice,
                             f->stream));
        CK(launch_forest_apply(f->x.p, x_dtype == SKNNR_F32, f->n_features, rows, f->n_features, f->d_nodes,
                               f->d_roots, f->n_trees, nullptr, f->ids.p, f->n_trees, f->stream));
        CK(cudaMemcpyAsync(out_ids + r0 * f->n_trees, f->ids.p, (size_t)rows * f->n_trees * 4, cudaMemcpyDeviceToHost,
                           f->stream));
        CK(cudaStreamSynchronize(f->stream));
    }
    return SKNNR_OK;
}

int sknnr_hamming_weighted_average(sknnr_hamming_index *ix, const int64_t *idx, const double *w,
                                   int64_t n_q, int32_t k, double *out_pred) {
    return weighted_average_common(ix, idx, w, n_q, k, out_pred);
}

// -----------------------------------------------------------------------------------------
int sknnr_measure_fp32_peak(int32_t device, double *tflops) {
    if (!tflops) return fail(SKNNR_EINVAL, "NULL argument");
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
        return fail(SKNNR_ENODEV, "no CUDA device");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    float *sink = nullptr;
    CK(cudaMalloc(&sink, 4));
    const int grid = prop.multiProcessorCount * 8, iters = 20000;
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    CK(launch_fp32_peak(sink, 1000, grid, 0));  // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 3; ++rep) {
        CK(cudaEventRecord(a, 0));
        CK(launch_fp32_peak(sink, iters, grid, 0));
        CK(cudaEventRecord(b, 0));
        CK(cudaEventSynchronize(b));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, a, b));
        const double flops = (double)grid * 256 * iters * 4 * 8 * 2 * 2;  // FFMA2 = 2 FMA = 4 FLOP
        best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(sink);
    *tflops = best;
    return SKNNR_OK;
}

}  // extern "C"

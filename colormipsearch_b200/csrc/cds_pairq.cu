// cds_pairq.cu -- the single-pair API of the reference, made usable on a GPU: a micro-batching scorer with a device-side target cache.
//
// The reference's provider interface is one call per (mask, target) pair --
// ColorDepthSearchAlgorithm.calculateMatchingScore(target, variantSuppliers)
// (colormipsearch-api/src/main/java/org/janelia/colormipsearch/cds/ColorDepthSearchAlgorithm.java:60-61) -- made from ~40 pool
// threads at once on one shared algorithm instance per mask
// (colormipsearch-tools/src/main/java/org/janelia/colormipsearch/cmd/cdsprocess/LocalColorMIPSearchProcessor.java:93-105), with
// the SAME target ImageArray object recurring across masks because targets come out of a Guava cache
// (colormipsearch-tools/.../cmd/CachedMIPsUtils.java:60-110).  A literal translation (upload 2 MB, encode, one tiny kernel,
// synchronise, per call and under a lock) loses to the CPU.  Here the calls of all threads meet in a queue:
//
//   * cds_pairq_score blocks its caller like the Java method does.  If the target's key (the caller's identity of the image: the
//     cache key or System.identityHashCode) is not in the device cache, the CALLING thread uploads and encodes it -- the copies of
//     different callers run in parallel and never pass through the dispatcher -- and leaves an event behind.
//   * one dispatcher thread per device collects what has arrived (up to max_batch requests, waiting at most max_wait_us for
//     company), launches ONE kernel for the whole batch, reads the score words back and wakes the callers.
//   * the kernel (pair_gather_kernel) scores a list of (mask, cache slot) pairs: kPairSplit CTAs per pair, each thread keeps the
//     counts of all shift / mirror variants of its mask pixels in registers (one record load for 18 gathers), partial counts meet in
//     global memory and the last CTA of a pair takes the maxima -- PixelMatchColorDepthSearchAlgorithm.java:166-263, bit for bit the
//     scores of the batched kernels (tests/test_pairq_gpu.py).
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <shared_mutex>
#include <deque>
#include <list>
#include <thread>
#include <unordered_map>

#include <climits>
#include <linux/futex.h>
#include <sys/syscall.h>
#include <unistd.h>

#include "cds_runtime.h"

using namespace cds;

namespace {

constexpr int kPairSplit = 4;            // CTAs per pair
constexpr int kPairThreads = 256;

__device__ __forceinline__ bool pair_code_matches(uint32_t c, uint32_t lo1, uint32_t len1, uint32_t lo2, uint32_t len2)
{
    return (c - lo1 <= len1) | (c - lo2 <= len2);
}

// The pairs of a launch travel in the kernel's parameter space (no copy to enqueue), the score words are written straight into
// pinned host memory the dispatcher reads after the stream has drained (no copy back), and the last CTA of a pair leaves the
// pair's accumulators zero for the next launch (no memset): a batch is ONE launch and one synchronisation.
constexpr int kPairsPerLaunch = 128;
constexpr int32_t kScorePending = -1;     // a score word is a count below 2^24 plus the mirror bit: never all ones
constexpr int kIdleSpinUs = 30;          // how long an idle dispatcher polls before it goes to sleep
inline void cpu_relax()
{
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#else
    std::this_thread::yield();
#endif
}
struct PairList {
    int32_t mask[kPairsPerLaunch];
    int32_t slot[kPairsPerLaunch];
};

// acc: [kPairsPerLaunch][2 * NV + 1], zero on entry and on exit (the last word counts the pair's finished CTAs); scores[pair] = score word
template <int NV>
__global__ void __launch_bounds__(kPairThreads) pair_gather_kernel(const MaskDesc *__restrict__ masks, const PairList pairs,
                                                                   const uint32_t *__restrict__ planes,
                                                                   PlaneGeom g, ShiftSet shifts, int *__restrict__ acc, int32_t *__restrict__ scores)
{
    __shared__ int s_cnt[2 * NV];
    __shared__ int s_last;
    const int pr = blockIdx.x, part = blockIdx.y;
    const MaskDesc md = masks[pairs.mask[pr]];
    const uint32_t *plane = planes + g.row_offset(pairs.slot[pr], 0);
    const int n_orient = shifts.mirror ? 2 : 1;
    int cnt[2 * NV];
#pragma unroll
    for (int v = 0; v < 2 * NV; v++) cnt[v] = 0;
    if (threadIdx.x < 2 * NV) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    for (int i = part * kPairThreads + threadIdx.x; i < md.P; i += kPairSplit * kPairThreads) {
        const uint4 q = __ldg(reinterpret_cast<const uint4 *>(md.records + i));
        const int x0 = (int) (q.x & 0xFFFFu), y0 = (int) (q.x >> 16);
        const uint32_t len1 = ((q.w & 0xFFFFu) << CDS_CODE_SR_SHIFT) | 0xFFu;
        const uint32_t len2 = ((q.w >> 16) << CDS_CODE_SR_SHIFT) | 0xFFu;
#pragma unroll
        for (int v = 0; v < NV; v++) {
            if (v >= shifts.n) break;
            const int x = x0 + shifts.dx[v], y = y0 + shifts.dy[v];
            if (x < 0 || x >= g.W || y < 0 || y >= g.H) continue;                      // shiftMaskPosArray :138-141
            const uint32_t *row = plane + (size_t) y * g.pitch;
            cnt[v] += pair_code_matches(__ldg(row + x), q.y, len1, q.z, len2) ? 1 : 0;
            if (n_orient == 2) cnt[NV + v] += pair_code_matches(__ldg(row + (g.W - 1 - x)), q.y, len1, q.z, len2) ? 1 : 0;   // mirrorMask :153-154 (after the shift)
        }
    }
#pragma unroll
    for (int v = 0; v < 2 * NV; v++) {
        const int c = __reduce_add_sync(0xffffffffu, cnt[v]);
        if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_cnt[v], c);
    }
    __syncthreads();
    const int stride = 2 * NV + 1;
    int *pacc = acc + (size_t) pr * stride;
    if (threadIdx.x < 2 * NV && s_cnt[threadIdx.x]) atomicAdd(&pacc[threadIdx.x], s_cnt[threadIdx.x]);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&pacc[2 * NV], 1) == kPairSplit - 1;
    __syncthreads();
    if (!s_last || threadIdx.x != 0) return;
    __threadfence();
    int best = 0, bestm = 0;
    for (int v = 0; v < shifts.n; v++) {
        best = max(best, __ldcg(&pacc[v]));
        bestm = max(bestm, __ldcg(&pacc[NV + v]));
    }
    int word = best;
    if (n_orient == 2 && bestm > best) word = bestm | CDS_SCORE_MIRROR_BIT;            // strict :189
    scores[pr] = word;
    for (int v = 0; v <= 2 * NV; v++) __stcg(&pacc[v], 0);
}

struct PairRequest {
    int32_t mask = 0, slot = -1;
    cudaEvent_t ready = nullptr;         // the slot's upload + encode (nullptr: already resident)
    int32_t word = 0;
    cds_status status = CDS_OK;
    std::atomic<bool> done{false};
};

// Callers sleep on the device's batch counter (a futex word) instead of a condition variable: one FUTEX_WAKE releases all callers
// of a batch at once and none of them has to take a mutex on the way out (40 threads re-acquiring one mutex one after the other
// were half of a batch's latency).
inline void futex_wait_u32(std::atomic<uint32_t> *addr, uint32_t expected)
{
    syscall(SYS_futex, reinterpret_cast<uint32_t *>(addr), FUTEX_WAIT_PRIVATE, expected, nullptr, nullptr, 0);
}
inline void futex_wake_all(std::atomic<uint32_t> *addr)
{
    syscall(SYS_futex, reinterpret_cast<uint32_t *>(addr), FUTEX_WAKE_PRIVATE, INT_MAX, nullptr, nullptr, 0);
}
// (Measured and dropped: callers sleeping in eight groups, the dispatcher waking one sleeper per group and every woken thread waking the
// rest of its group.  The callers then come back staggered, batches shrink from 40 to 34 requests, and 40 / 80 threads reach 414 k / 213 k
// pairs/s instead of 515 k / 589 k with the one broadcast.)

struct CacheSlot {
    uint64_t key = 0;
    int refs = 0;                        // requests in flight that use the slot
    bool valid = false;
    bool loading = false;                // a caller is uploading the slot's image right now
    cudaEvent_t ready = nullptr;         // recorded after the slot's encode; kept while the slot is valid
    bool ready_pending = false;          // the event may not have completed yet
    std::list<int>::iterator lru;
};

struct PairDev {
    int d = 0;                           // index into ctx->devs
    cudaStream_t stream = nullptr;       // dispatcher's stream
    uint32_t *planes = nullptr;          // [n_slots] code planes
    std::vector<CacheSlot> slots;
    std::list<int> lru;                  // least recently used first
    std::unordered_map<uint64_t, int> by_key;
    std::deque<PairRequest *> queue;
    std::atomic<int> queued{0};          // queue.size(), readable without the mutex (the dispatcher polls it while it waits for company)
    std::atomic<bool> disp_sleeping{false};     // the dispatcher sleeps on cv_work: only then does a push pay for a notify
    std::mutex mu;
    std::condition_variable cv_work, cv_slot;
    std::atomic<uint32_t> generation{0};  // batches completed: what callers sleep on
    std::thread worker;
    bool busy = false;                   // the dispatcher is between taking a batch and finishing it
    std::condition_variable cv_idle;
    // upload staging: one device buffer + stream + pinned host buffer per upload lane (callers take a lane for the length of an upload)
    struct Lane { cudaStream_t stream = nullptr; uint8_t *d_rgb = nullptr; uint8_t *h_rgb = nullptr; bool busy = false; };
    std::vector<Lane> lanes;
    // batch buffers
    int32_t *h_scores = nullptr, *d_scores_alias = nullptr;      // pinned + mapped: the kernel writes, the dispatcher reads
    int *d_acc = nullptr;
    int64_t batches = 0, requests = 0, uploads = 0;
};

}  // namespace

struct cds_pairq {
    cds_ctx *ctx = nullptr;
    const cds_maskset *ms = nullptr;
    PlaneGeom g{};
    int max_batch = 64;
    int max_wait_us = 50;
    std::vector<std::unique_ptr<PairDev>> devs;
    std::atomic<bool> stop{false};
    std::atomic<uint64_t> anon{0};
    // masks may be added to the mask set while the queue exists (one provider, one queue, an algorithm per mask): a call that names a
    // mask the queue has not seen quiesces the dispatchers, rebuilds the device descriptors and goes on
    std::atomic<int> n_masks{0};
    std::vector<int32_t> sizes;          // getQuerySize() of the masks the queue knows (a private copy: the mask set's vector may grow)
    std::shared_mutex refresh_mu;        // readers (every call) share it; a refresh takes it alone
};

namespace {

// pairs [first, first + n) of the batch (n <= kPairsPerLaunch); consecutive launches of a batch share the accumulators in stream order
void launch_pair_gather(const cds_pairq *q, PairDev &pd, const PairList &pl, int first, int n, const MaskDesc *descs)
{
    const ShiftSet &sh = q->ms->shifts;
    const dim3 grid((unsigned) n, kPairSplit);
    const int nv = sh.n <= 1 ? 1 : (sh.n <= 9 ? 9 : (sh.n <= 17 ? 17 : CDS_MAX_SHIFT_OFFSETS));
    int32_t *out = pd.d_scores_alias + first;
    if (nv == 1) pair_gather_kernel<1><<<grid, kPairThreads, 0, pd.stream>>>(descs, pl, pd.planes, q->g, sh, pd.d_acc, out);
    else if (nv == 9) pair_gather_kernel<9><<<grid, kPairThreads, 0, pd.stream>>>(descs, pl, pd.planes, q->g, sh, pd.d_acc, out);
    else if (nv == 17) pair_gather_kernel<17><<<grid, kPairThreads, 0, pd.stream>>>(descs, pl, pd.planes, q->g, sh, pd.d_acc, out);
    else pair_gather_kernel<CDS_MAX_SHIFT_OFFSETS><<<grid, kPairThreads, 0, pd.stream>>>(descs, pl, pd.planes, q->g, sh, pd.d_acc, out);
}

void dispatcher(cds_pairq *q, PairDev *pdp)
{
    PairDev &pd = *pdp;
    cds_ctx *ctx = q->ctx;
    cudaSetDevice(ctx->devs[pd.d].dev);
    std::vector<PairRequest *> batch;
    int last_n = 1;
    for (;;) {
        batch.clear();
        {
            // Nothing queued: poll for a moment (the callers of the batch that has just been answered are on their way back), then
            // sleep.  Polling reads one atomic counter and takes no lock, so it does not stand in the callers' way.
            if (pd.queued.load(std::memory_order_acquire) == 0 && !q->stop.load()) {
                const auto spin_until = std::chrono::steady_clock::now() + std::chrono::microseconds(kIdleSpinUs);
                while (pd.queued.load(std::memory_order_acquire) == 0 && !q->stop.load() && std::chrono::steady_clock::now() < spin_until) cpu_relax();
            }
            if (pd.queued.load(std::memory_order_acquire) == 0) {
                std::unique_lock<std::mutex> lk(pd.mu);
                pd.disp_sleeping.store(true, std::memory_order_seq_cst);
                pd.cv_work.wait(lk, [&] { return q->stop.load() || !pd.queue.empty(); });
                pd.disp_sleeping.store(false, std::memory_order_seq_cst);
                if (pd.queue.empty() && q->stop.load()) return;
            }
            // wait a little for company: a batch of one costs the same launch and round trip as a batch of sixty-four
            // (as many as came last time -- the callers are a pool of threads that come back together -- or the deadline)
            const int expect = std::min(q->max_batch, std::max(1, last_n));
            if (pd.queued.load(std::memory_order_acquire) < expect && q->max_wait_us > 0) {
                const auto deadline = std::chrono::steady_clock::now() + std::chrono::microseconds(q->max_wait_us);
                while (pd.queued.load(std::memory_order_acquire) < expect && !q->stop.load() && std::chrono::steady_clock::now() < deadline) cpu_relax();
            }
            std::unique_lock<std::mutex> lk(pd.mu);
            while (!pd.queue.empty() && (int) batch.size() < q->max_batch) { batch.push_back(pd.queue.front()); pd.queue.pop_front(); }
            pd.queued.store((int) pd.queue.size(), std::memory_order_release);
            pd.busy = !batch.empty();
        }
        const int n = (int) batch.size();
        if (n == 0) continue;
        last_n = n;
        cudaError_t e = cudaSuccess;
        // the kernel writes every pair's score word into mapped host memory: a word that no score can be marks "not yet"
        volatile int32_t *hs = pd.h_scores;
        for (int i = 0; i < n; i++) hs[i] = kScorePending;
        for (int i = 0; i < n; i++)
            if (batch[i]->ready && e == cudaSuccess) e = cudaStreamWaitEvent(pd.stream, batch[i]->ready, 0);
        for (int first = 0; first < n && e == cudaSuccess; first += kPairsPerLaunch) {
            const int cnt = std::min(kPairsPerLaunch, n - first);
            PairList pl;
            for (int i = 0; i < cnt; i++) { pl.mask[i] = batch[first + i]->mask; pl.slot[i] = batch[first + i]->slot; }
            for (int i = cnt; i < kPairsPerLaunch; i++) { pl.mask[i] = 0; pl.slot[i] = 0; }
            launch_pair_gather(q, pd, pl, first, cnt, q->ms->d_descs[pd.d]);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) {
            // wait for the words themselves (a microsecond after the kernel's last store) rather than for the stream; every 200 us of
            // waiting the stream is asked whether it failed
            auto next_query = std::chrono::steady_clock::now() + std::chrono::microseconds(200);
            for (int i = 0; i < n && e == cudaSuccess; i++) {
                while (hs[i] == kScorePending) {
                    cpu_relax();
                    if (std::chrono::steady_clock::now() >= next_query) {
                        const cudaError_t qe = cudaStreamQuery(pd.stream);
                        if (qe == cudaSuccess) { if (hs[i] == kScorePending) e = cudaErrorUnknown; break; }     // finished without writing: cannot happen
                        if (qe != cudaErrorNotReady) { e = qe; break; }
                        next_query = std::chrono::steady_clock::now() + std::chrono::microseconds(200);
                    }
                }
            }
            std::atomic_thread_fence(std::memory_order_acquire);
        }
        if (e != cudaSuccess) { cudaStreamSynchronize(pd.stream); cudaGetLastError(); }
        {
            std::lock_guard<std::mutex> lk(pd.mu);
            pd.batches++;
            pd.requests += n;
            for (int i = 0; i < n; i++) {
                PairRequest *r = batch[i];
                r->word = e == cudaSuccess ? pd.h_scores[i] : 0;
                r->status = e == cudaSuccess ? CDS_OK : CDS_ERR_CUDA;
                CacheSlot &cs = pd.slots[r->slot];
                cs.ready_pending = false;            // the batch ran behind the slot's event
                if (--cs.refs == 0) pd.cv_slot.notify_all();
            }
            pd.busy = false;
        }
        pd.cv_idle.notify_all();
        for (int i = 0; i < n; i++) batch[i]->done.store(true, std::memory_order_release);      // (the request lives on its caller's stack: not touched after this)
        pd.generation.fetch_add(1, std::memory_order_release);
        futex_wake_all(&pd.generation);
    }
}

}  // namespace

extern "C" cds_status cds_pairq_create(cds_ctx *ctx, const cds_maskset *ms, int32_t max_batch, int32_t max_wait_us, int32_t cache_targets,
                                       cds_pairq **out)
{
    return cds::abi_guard("cds_pairq_create", [&]() -> cds_status {
        if (!ctx || !ms || !out) { set_tls_error("cds_pairq_create: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        *out = nullptr;
        if (ms->ctx != ctx) return ctx->fail(CDS_ERR_BAD_ARG, "cds_pairq_create: mask set belongs to another context");
        if (max_batch <= 0) max_batch = 64;
        if (max_batch > 4096) max_batch = 4096;
        if (max_wait_us < 0) max_wait_us = 0;
        if (cache_targets < 2 * max_batch) cache_targets = 2 * max_batch;          // a batch's slots are pinned while it runs
        cds_status st = const_cast<cds_maskset *>(ms)->sync_descs();
        if (st != CDS_OK) return st;
        std::unique_ptr<cds_pairq> q(new cds_pairq());
        q->ctx = ctx; q->ms = ms; q->max_batch = max_batch; q->max_wait_us = max_wait_us;
        q->g.W = ms->W; q->g.H = ms->H; q->g.pitch = choose_pitch(ms->W); q->g.guard = CDS_GUARD_ROWS;
        q->sizes = ms->sizes;
        q->n_masks.store((int) ms->sizes.size());
        const size_t img_bytes = (size_t) ms->W * ms->H * 3;
        const int nv_max = 2 * CDS_MAX_SHIFT_OFFSETS + 1;
        // Several independent queues per device (targets are spread over them by key, each has its share of the cache, its stream and its
        // dispatcher): a batch's turn-around is dominated by waking its callers and letting them back in, which costs ~1 us per caller ON
        // TOP of ~35 us per batch, so several batches of a few in flight answer more calls per second than one batch of forty.
        // (default: a third of the host's hardware threads, 2 .. 8 -- every queue has a dispatcher thread that polls for a moment before it
        // sleeps; measured on 16 cores: 40 / 80 callers reach 505 k / 660 k pairs/s with one queue, 500 k / 820 k with four, 520-580 k /
        // 870-900 k with six or eight, and lose with twelve or more)
        static const int queues_auto = (int) std::max(2u, std::min(8u, std::thread::hardware_concurrency() / 3u));
        static const int queues_per_dev = std::max(1, std::min(16, std::getenv("CDSGPU_PAIRQ_QUEUES") ? std::atoi(std::getenv("CDSGPU_PAIRQ_QUEUES")) : queues_auto));
        const int n_lanes = std::max(2, 8 / queues_per_dev);
        cache_targets = std::max(2 * max_batch, (cache_targets + queues_per_dev - 1) / queues_per_dev);
        for (size_t dq = 0; dq < ctx->devs.size() * (size_t) queues_per_dev && st == CDS_OK; dq++) {
            const size_t d = dq / (size_t) queues_per_dev;
            std::unique_ptr<PairDev> pd(new PairDev());
            pd->d = (int) d;
            st = ctx->check(cudaSetDevice(ctx->devs[d].dev), "cudaSetDevice");
            if (st == CDS_OK) st = ctx->check(cudaStreamCreateWithFlags(&pd->stream, cudaStreamNonBlocking), "cudaStreamCreate");
            const size_t words = q->g.total_words(cache_targets);
            if (st == CDS_OK) st = ctx->check(cudaMalloc(&pd->planes, words * sizeof(uint32_t)), "cudaMalloc(pair cache)");
            if (st == CDS_OK) { launch_fill_words(pd->planes, words, CDS_CODE_PAD_WORD, pd->stream); st = ctx->check(cudaGetLastError(), "fill"); }
            pd->slots.resize(cache_targets);
            for (int s = 0; s < cache_targets && st == CDS_OK; s++) {
                st = ctx->check(cudaEventCreateWithFlags(&pd->slots[s].ready, cudaEventDisableTiming), "cudaEventCreate");
                pd->lru.push_back(s);
                pd->slots[s].lru = std::prev(pd->lru.end());
            }
            pd->lanes.resize(n_lanes);
            for (int l = 0; l < n_lanes && st == CDS_OK; l++) {
                st = ctx->check(cudaStreamCreateWithFlags(&pd->lanes[l].stream, cudaStreamNonBlocking), "cudaStreamCreate");
                if (st == CDS_OK) st = ctx->check(cudaMalloc(&pd->lanes[l].d_rgb, img_bytes + 64), "cudaMalloc(pair staging)");
                if (st == CDS_OK) st = ctx->check(cudaHostAlloc(&pd->lanes[l].h_rgb, img_bytes, cudaHostAllocDefault), "cudaHostAlloc(pair staging)");
            }
            if (st == CDS_OK) st = ctx->check(cudaMalloc(&pd->d_acc, (size_t) kPairsPerLaunch * nv_max * sizeof(int)), "cudaMalloc");
            if (st == CDS_OK) st = ctx->check(cudaMemsetAsync(pd->d_acc, 0, (size_t) kPairsPerLaunch * nv_max * sizeof(int), pd->stream), "memset");
            if (st == CDS_OK) st = ctx->check(cudaHostAlloc(&pd->h_scores, (size_t) max_batch * sizeof(int32_t), cudaHostAllocMapped), "cudaHostAlloc");
            if (st == CDS_OK) st = ctx->check(cudaHostGetDevicePointer((void **) &pd->d_scores_alias, pd->h_scores, 0), "cudaHostGetDevicePointer");
            if (st == CDS_OK) st = ctx->check(cudaStreamSynchronize(pd->stream), "pair cache");
            q->devs.push_back(std::move(pd));
        }
        if (st != CDS_OK) { cds_pairq_destroy(q.release()); return st; }
        for (auto &pd : q->devs) pd->worker = std::thread(dispatcher, q.get(), pd.get());
        *out = q.release();
        return CDS_OK;
    });
}

extern "C" void cds_pairq_destroy(cds_pairq *q)
{
    if (!q) return;
    q->stop.store(true);
    for (auto &pd : q->devs) {
        { std::lock_guard<std::mutex> lk(pd->mu); }
        pd->cv_work.notify_all();
        if (pd->worker.joinable()) pd->worker.join();
        cudaSetDevice(q->ctx->devs[pd->d].dev);
        if (pd->stream) { cudaStreamSynchronize(pd->stream); cudaStreamDestroy(pd->stream); }
        for (auto &l : pd->lanes) {
            if (l.stream) { cudaStreamSynchronize(l.stream); cudaStreamDestroy(l.stream); }
            if (l.d_rgb) cudaFree(l.d_rgb);
            if (l.h_rgb) cudaFreeHost(l.h_rgb);
        }
        for (auto &s : pd->slots) if (s.ready) cudaEventDestroy(s.ready);
        for (void *p : {(void *) pd->planes, (void *) pd->d_acc}) if (p) cudaFree(p);
        if (pd->h_scores) cudaFreeHost(pd->h_scores);
    }
    cudaGetLastError();
    delete q;
}

extern "C" cds_status cds_pairq_score(cds_pairq *q, int32_t mask_index, uint64_t target_key, const uint8_t *target_rgb,
                                      int32_t target_width, int32_t target_height,
                                      int32_t *score_out, double *ratio_out, int32_t *mirrored_out)
{
    return cds::abi_guard("cds_pairq_score", [&]() -> cds_status {
        if (!q || !score_out || !ratio_out || !mirrored_out) { set_tls_error("cds_pairq_score: NULL argument"); return CDS_ERR_BAD_ARG; }
        const cds_maskset *ms = q->ms;
        if (mask_index >= q->n_masks.load(std::memory_order_acquire) && mask_index >= 0) {
            // a mask added after the queue was created: stop the dispatchers between two batches, rebuild the descriptors, go on
            std::unique_lock<std::shared_mutex> rl(q->refresh_mu);
            if (mask_index >= q->n_masks.load()) {
                std::lock_guard<std::recursive_mutex> cl(q->ctx->mu);
                if (mask_index < (int) ms->sizes.size()) {
                    std::vector<std::unique_lock<std::mutex>> held;
                    for (auto &pd : q->devs) {
                        held.emplace_back(pd->mu);
                        pd->cv_idle.wait(held.back(), [&] { return !pd->busy; });
                    }
                    const cds_status rs = const_cast<cds_maskset *>(ms)->sync_descs();
                    if (rs != CDS_OK) return rs;
                    q->sizes = ms->sizes;                      // (callers read q->sizes only below n_masks, and never while it is replaced: see below)
                    q->n_masks.store((int) ms->sizes.size(), std::memory_order_release);
                }
            }
        }
        if (mask_index < 0 || mask_index >= q->n_masks.load(std::memory_order_acquire)) { set_tls_error("cds_pairq_score: mask index out of range"); return CDS_ERR_BAD_ARG; }
        int P;
        {
            std::shared_lock<std::shared_mutex> rl(q->refresh_mu);     // short: guards the vector against a concurrent refresh
            P = q->sizes[mask_index];
        }
        if (P == 0) { *score_out = 0; *ratio_out = 0; *mirrored_out = 0; return CDS_OK; }   // PixelMatch...:169-170 (before the size check)
        if (target_width != ms->W || target_height != ms->H) {
            char buf[200];
            snprintf(buf, sizeof buf, "Invalid image size - target's image size (%d, %d) must match query's image size: (%d, %d)",
                     ms->W, ms->H, target_width, target_height);
            set_tls_error(buf);
            return CDS_ERR_SIZE_MISMATCH;
        }
        if (!target_rgb) { set_tls_error("cds_pairq_score: target is NULL"); return CDS_ERR_BAD_ARG; }
        const bool anonymous = target_key == 0;
        if (anonymous) target_key = 0x8000000000000000ull | ++q->anon;                    // never found again: a one-shot slot
        PairDev &pd = *q->devs[(size_t) (target_key % q->devs.size())];
        cds_ctx *ctx = q->ctx;
        const size_t img_bytes = (size_t) ms->W * ms->H * 3;
        PairRequest req;
        req.mask = mask_index;
        int lane = -1;
        bool pushed = false;                 // a resident target: the request is queued inside the lookup's critical section
        {
            std::unique_lock<std::mutex> lk(pd.mu);
            for (;;) {
                auto it = anonymous ? pd.by_key.end() : pd.by_key.find(target_key);
                if (it != pd.by_key.end()) {
                    req.slot = it->second;
                    CacheSlot &cs = pd.slots[req.slot];
                    cs.refs++;                                   // pins the slot while we wait for another caller's upload of the same image
                    pd.cv_slot.wait(lk, [&] { return !cs.loading; });
                    cs.refs--;
                    if (!cs.valid) { set_tls_error("cds_pairq_score: the upload of this target failed in another thread"); return CDS_ERR_CUDA; }
                    if (cs.ready_pending) req.ready = cs.ready;
                    break;
                }
                // a free slot (least recently used, not referenced by a request in flight) and an upload lane
                int victim = -1;
                for (int s : pd.lru) if (pd.slots[s].refs == 0) { victim = s; break; }
                if (victim >= 0) {
                    for (size_t l = 0; l < pd.lanes.size(); l++) if (!pd.lanes[l].busy) { lane = (int) l; break; }
                    if (lane >= 0) { req.slot = victim; break; }
                }
                // none yet: wait, then look the key up again -- another caller may have started uploading this image meanwhile
                pd.cv_slot.wait(lk);
            }
            if (lane >= 0) {
                CacheSlot &cs = pd.slots[req.slot];
                auto old = pd.by_key.find(cs.key);
                if (old != pd.by_key.end() && old->second == req.slot) pd.by_key.erase(old);
                cs.key = target_key; cs.valid = false; cs.loading = true;
                if (!anonymous) pd.by_key[target_key] = req.slot;      // later callers with this image wait for this upload
                pd.lanes[lane].busy = true;
                pd.uploads++;
            }
            CacheSlot &cs = pd.slots[req.slot];
            cs.refs++;
            pd.lru.splice(pd.lru.end(), pd.lru, cs.lru);       // most recently used (the iterator stays valid)
            if (lane < 0) {
                pd.queue.push_back(&req);
                pd.queued.store((int) pd.queue.size(), std::memory_order_release);
                pushed = true;
            }
        }
        cds_status st = CDS_OK;
        if (lane >= 0) {
            // this thread uploads and encodes its target: through its lane's pinned buffer, on its lane's stream
            PairDev::Lane &ln = pd.lanes[lane];
            cudaError_t e = cudaSetDevice(ctx->devs[pd.d].dev);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ln.stream);                    // the lane's previous upload has left the pinned buffer
            if (e == cudaSuccess) {
                memcpy(ln.h_rgb, target_rgb, img_bytes);
                e = cudaMemcpyAsync(ln.d_rgb, ln.h_rgb, img_bytes, cudaMemcpyHostToDevice, ln.stream);
            }
            if (e == cudaSuccess) {
                launch_encode_rgb(ln.d_rgb, 1, pd.planes, q->g, req.slot, ctx->devs[pd.d].d_rank_tab, ms->params.data_threshold, ln.stream);
                e = cudaGetLastError();
            }
            CacheSlot &cs = pd.slots[req.slot];
            if (e == cudaSuccess) e = cudaEventRecord(cs.ready, ln.stream);
            std::lock_guard<std::mutex> lk(pd.mu);
            ln.busy = false;
            cs.loading = false;
            if (e == cudaSuccess) {
                cs.valid = true; cs.ready_pending = true;
                req.ready = cs.ready;
            } else {
                cudaGetLastError();
                st = CDS_ERR_CUDA;
                set_tls_error(std::string("cds_pairq_score: upload failed: ") + cudaGetErrorString(e));
                auto mine = pd.by_key.find(target_key);
                if (mine != pd.by_key.end() && mine->second == req.slot) pd.by_key.erase(mine);
                cs.refs--;
            }
            pd.cv_slot.notify_all();
        }
        if (st != CDS_OK) return st;
        if (!pushed) {
            std::lock_guard<std::mutex> lk(pd.mu);
            pd.queue.push_back(&req);
            pd.queued.store((int) pd.queue.size(), std::memory_order_release);
        }
        if (pd.disp_sleeping.load(std::memory_order_seq_cst)) pd.cv_work.notify_one();
        for (;;) {
            const uint32_t g = pd.generation.load(std::memory_order_acquire);
            if (req.done.load(std::memory_order_acquire)) break;
            futex_wait_u32(&pd.generation, g);
        }
        if (req.status != CDS_OK) { set_tls_error("cds_pairq_score: the batch's kernel failed"); return req.status; }
        *score_out = req.word & ~CDS_SCORE_MIRROR_BIT;
        *mirrored_out = (req.word & CDS_SCORE_MIRROR_BIT) ? 1 : 0;
        *ratio_out = (double) *score_out / (double) P;     // :194
        return CDS_OK;
    });
}

extern "C" cds_status cds_pairq_get_stats(const cds_pairq *q, int64_t *requests, int64_t *batches, int64_t *uploads)
{
    if (!q) { set_tls_error("cds_pairq_get_stats: NULL queue"); return CDS_ERR_BAD_ARG; }
    int64_t r = 0, b = 0, u = 0;
    for (auto &pd : q->devs) {
        std::lock_guard<std::mutex> lk(pd->mu);
        r += pd->requests; b += pd->batches; u += pd->uploads;
    }
    if (requests) *requests = r;
    if (batches) *batches = b;
    if (uploads) *uploads = u;
    return CDS_OK;
}


// Test / bench hook: drives cds_pairq_score from n_threads native threads the way the reference's thread pool drives
// calculateMatchingScore (each thread takes the next pair of the list, blocks in the call, stores the result), so that the
// throughput of the single-pair entry point can be measured without an interpreter lock in the way.  Target image t has key
// keys[t] (0 = no caching).  seconds_out = wall clock of the whole run.
extern "C" cds_status cds_debug_pairq_drive(cds_pairq *q, const uint8_t *targets_rgb, int64_t n_targets, const uint64_t *keys,
                                            const int32_t *pair_mask, const int64_t *pair_target, int64_t n_pairs, int32_t n_threads,
                                            int32_t *scores_out, uint8_t *mirrored_out, double *seconds_out)
{
    return cds::abi_guard("cds_debug_pairq_drive", [&]() -> cds_status {
        if (!q || !targets_rgb || !pair_mask || !pair_target || !scores_out || !seconds_out || n_threads <= 0 || n_pairs < 0) {
            set_tls_error("cds_debug_pairq_drive: bad arguments");
            return CDS_ERR_BAD_ARG;
        }
        for (int64_t i = 0; i < n_pairs; i++)
            if (pair_target[i] < 0 || pair_target[i] >= n_targets) { set_tls_error("cds_debug_pairq_drive: target index out of range"); return CDS_ERR_BAD_ARG; }
        const size_t img_bytes = (size_t) q->ms->W * q->ms->H * 3;
        std::atomic<int64_t> next{0};
        std::atomic<int> failed{0};
        auto body = [&]() {
            for (;;) {
                const int64_t i = next.fetch_add(1);
                if (i >= n_pairs) return;
                int32_t sc = 0, mir = 0;
                double ratio = 0;
                const int64_t t = pair_target[i];
                const cds_status st = cds_pairq_score(q, pair_mask[i], keys ? keys[t] : 0, targets_rgb + (size_t) t * img_bytes, q->ms->W, q->ms->H, &sc, &ratio, &mir);
                if (st != CDS_OK) { failed.store((int) st); return; }
                scores_out[i] = sc;
                if (mirrored_out) mirrored_out[i] = (uint8_t) mir;
            }
        };
        const auto t0 = std::chrono::steady_clock::now();
        std::vector<std::thread> pool;
        for (int t = 0; t < n_threads; t++) pool.emplace_back(body);
        for (auto &th : pool) th.join();
        *seconds_out = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        if (failed.load()) { set_tls_error("cds_debug_pairq_drive: a call failed"); return (cds_status) failed.load(); }
        return CDS_OK;
    });
}

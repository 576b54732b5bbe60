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
#include <cstdio>
#include <shared_mutex>

#include "cds_queue.h"

using namespace cds;

namespace {

constexpr int kPairSplit = 4;            // CTAs per pair
constexpr int kPairThreads = 256;

__device__ __forceinline__ bool pair_code_matches(uint32_t c, uint32_t lo1, uint32_t len1, uint32_t lo2, uint32_t len2)
{
    return (c - lo1 <= len1) | (c - lo2 <= len2);
}

// The score words are written straight into pinned host memory the dispatcher reads (no copy back), and the last CTA of a pair
// leaves the pair's accumulators zero for the next launch (no memset): a batch is ONE launch and one synchronisation.
constexpr int kPairsPerLaunch = pq::kPairsPerLaunch;
constexpr int32_t kScorePending = -1;     // a score word is a count below 2^24 plus the mirror bit: never all ones
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

struct PairRequest : pq::Request {
    int32_t word = 0;
};

struct PairDev : pq::Queue {
    uint32_t *planes = nullptr;          // [slots] code planes
    int32_t *h_scores = nullptr, *d_scores_alias = nullptr;      // pinned + mapped: the kernel writes, the dispatcher reads
    int *d_acc = nullptr;
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
    cudaSetDevice(q->ctx->devs[pd.d].dev);
    std::vector<pq::Request *> batch;
    int last_n = 1;
    while (pd.collect(batch, q->max_batch, q->max_wait_us, last_n, q->stop)) {
        const int n = (int) batch.size();
        // the kernel writes every pair's score word into mapped host memory: a word that no score can be marks "not yet"
        volatile int32_t *hs = pd.h_scores;
        for (int i = 0; i < n; i++) hs[i] = kScorePending;
        cudaError_t e = pd.wait_fills(batch);
        for (int first = 0; first < n && e == cudaSuccess; first += kPairsPerLaunch) {
            const int cnt = std::min(kPairsPerLaunch, n - first);
            PairList pl;
            for (int i = 0; i < cnt; i++) { pl.mask[i] = batch[first + i]->mask; pl.slot[i] = batch[first + i]->slot; }
            for (int i = cnt; i < kPairsPerLaunch; i++) { pl.mask[i] = 0; pl.slot[i] = 0; }
            launch_pair_gather(q, pd, pl, first, cnt, q->ms->d_descs[pd.d]);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = pd.await_results(n, [&](int i) { return hs[i] != kScorePending; });
        pd.complete(batch, e, [&](pq::Request *r, int i) { static_cast<PairRequest *>(r)->word = pd.h_scores[i]; });
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
        const pq::Plan plan = pq::plan(cache_targets, max_batch);
        for (size_t dq = 0; dq < ctx->devs.size() * (size_t) plan.queues_per_dev && st == CDS_OK; dq++) {
            const size_t d = dq / (size_t) plan.queues_per_dev;
            std::unique_ptr<PairDev> pd(new PairDev());
            st = ctx->check(cudaSetDevice(ctx->devs[d].dev), "cudaSetDevice");
            if (st == CDS_OK) st = pd->init(ctx, (int) d, plan.slots_per_queue, plan.lanes_per_queue, img_bytes);
            const size_t words = q->g.total_words(plan.slots_per_queue);
            if (st == CDS_OK) st = ctx->check(cudaMalloc(&pd->planes, words * sizeof(uint32_t)), "cudaMalloc(pair cache)");
            if (st == CDS_OK) { launch_fill_words(pd->planes, words, CDS_CODE_PAD_WORD, pd->stream); st = ctx->check(cudaGetLastError(), "fill"); }
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
        pd->stop_and_join();
        cudaSetDevice(q->ctx->devs[pd->d].dev);
        pd->release();
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
                    const cds_status rs = pq::quiesced(q->devs, [&]() -> cds_status {
                        const cds_status ss = const_cast<cds_maskset *>(ms)->sync_descs();
                        if (ss != CDS_OK) return ss;
                        q->sizes = ms->sizes;                  // (callers read q->sizes only below n_masks, and never while it is replaced: see below)
                        q->n_masks.store((int) ms->sizes.size(), std::memory_order_release);
                        return CDS_OK;
                    });
                    if (rs != CDS_OK) return rs;
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
        cds_status st = pd.acquire(req, target_key, anonymous, lane, "cds_pairq_score");
        if (st != CDS_OK) return st;
        if (lane >= 0) {
            // this thread uploads and encodes its target: through its lane's pinned buffer, on its lane's stream
            pq::Lane &ln = pd.lanes[lane];
            cudaError_t e = cudaSetDevice(ctx->devs[pd.d].dev);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ln.stream);                    // the lane's previous upload has left the pinned buffer
            if (e == cudaSuccess) {
                memcpy(ln.h_stage, target_rgb, img_bytes);
                e = cudaMemcpyAsync(ln.d_stage, ln.h_stage, img_bytes, cudaMemcpyHostToDevice, ln.stream);
            }
            if (e == cudaSuccess) {
                launch_encode_rgb(ln.d_stage, 1, pd.planes, q->g, req.slot, ctx->devs[pd.d].d_rank_tab, ms->params.data_threshold, ln.stream);
                e = cudaGetLastError();
            }
            if (e == cudaSuccess) e = cudaEventRecord(pd.slots[req.slot].ready, ln.stream);
            st = pd.filled(req, target_key, lane, e, "cds_pairq_score");
            if (st != CDS_OK) return st;
        }
        pd.wait(req);
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
    pq::sum_stats(q->devs, requests, batches, uploads);
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

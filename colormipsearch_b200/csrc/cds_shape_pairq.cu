// cds_shape_pairq.cu -- the shape score's single-pair call, made usable on a GPU: a micro-batching scorer with a device-side cache
// of derived target planes.
//
// gradientScores scores a mask's top lines through Shape2DMatchColorDepthSearchAlgorithm.calculateMatchingScore(target,
// variantSuppliers) (API/cds/Shape2DMatchColorDepthSearchAlgorithm.java:150-245), one blocking call per (mask, target) pair from a
// thread pool (TOOLS/CalculateGradientScoresCmd.java:304-312), and the same target recurs across masks because every mask scores its
// top lines out of one library.  The calls of all threads meet in the queue machinery of cds_queue.h:
//
//   * a slot of the cache holds one target's derived planes: the slice plane of its thresholded zgap image, its gradient and its
//     signal bitmap.  On a miss the CALLING thread fills the slot on its upload lane -- pinned staging, cudaMemcpyAsync, then the very
//     launches the batched call makes for one target (launch_shape_target_planes) -- and leaves an event behind.
//   * a dispatcher per queue collects what has arrived and launches shape_pair_batch_kernel once per 128 pairs: kShapePairSplit CTAs
//     per pair share its gap list and bitmap words, partial sums meet in global memory and the last CTA of a pair applies the mirror
//     rule and writes (gap, area, mirrored) into mapped host memory -- bit for bit what cds_shape_score_pairs returns
//     (tests/test_shape_pairq_gpu.py), since both kernels add the same per-pixel terms (cds_shape.cuh).
#include <cstdio>
#include <cstring>
#include <shared_mutex>

#include "cds_queue.h"
#include "cds_shape.cuh"

using namespace cds;

namespace {

// CTAs per pair.  A gradientScores-like batch is ~40 pairs: one CTA per pair (shape_pair_kernel's grid) would leave most of the 148 SMs
// idle.  Measured with tools/shape_pairq_bench.py (B200 at 1000 W, 64 masks x 300 of 512 resident targets, 1210 x 566), pairs/s from
// 8 / 40 native callers: 1 CTA 69 k / 285 k, 2: 108 k / 375 k, 4: 149 k / 559 k, 8: 184 k / 662 k, 16: 213 k / 621 k
// (profiles/shape_pairq_split_sweep.txt)
constexpr int kShapePairSplit = 8;
constexpr int kShapePairThreads = 256;
constexpr int kPairsPerLaunch = pq::kPairsPerLaunch;
constexpr int kAccWords = 5;               // per pair: gap, mirrored gap, area, mirrored area, finished CTAs
constexpr int32_t kResultPending = -1;     // a result's mirrored word is 0 or 1 once written

struct ShapePairList {
    int32_t mask[kPairsPerLaunch];
    int32_t slot[kPairsPerLaunch];
};

struct ShapePairResult {
    long long gap, he;
    int32_t mirrored;                      // written last, after a system-wide fence: the dispatcher polls it
    int32_t pad;
};

// acc: [kPairsPerLaunch][kAccWords], zero on entry and on exit; out[pair] in mapped host memory
__global__ void __launch_bounds__(kShapePairThreads) shape_pair_batch_kernel(const ShapeMaskDesc *__restrict__ masks, const ShapePairList pl,
                                                                             const uint16_t *__restrict__ zslice, const uint16_t *__restrict__ grad,
                                                                             const uint32_t *__restrict__ tsig, int W, int H, int bpitch, int mirror,
                                                                             unsigned long long *__restrict__ acc, ShapePairResult *out)
{
    __shared__ long long s_red[4][kShapePairThreads / 32];
    __shared__ int s_last;
    const int pr = blockIdx.x, part = blockIdx.y, split = (int) gridDim.y;
    const int64_t t = pl.slot[pr];
    const ShapeMaskDesc md = masks[pl.mask[pr]];
    const uint16_t *zs = zslice + (size_t) t * W * H;
    const uint16_t *gr = grad + (size_t) t * W * H;
    const uint32_t *ts = tsig + (size_t) t * H * bpitch;
    const int stride = split * kShapePairThreads;
    long long gap_n = 0, gap_m = 0, he_n = 0, he_m = 0;
    for (int i = part * kShapePairThreads + threadIdx.x; i < md.n_gap; i += stride) shape_gap_entry(__ldg(md.gap_list + i), zs, gr, W, mirror, gap_n, gap_m);
    const int n_words = H * bpitch;
    for (int i = part * kShapePairThreads + threadIdx.x; i < n_words; i += stride) shape_he_word(md, ts, i, mirror, he_n, he_m);
    long long v[4] = {gap_n, gap_m, he_n, he_m};
#pragma unroll
    for (int k = 0; k < 4; k++) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], off);
        if ((threadIdx.x & 31) == 0) s_red[k][threadIdx.x >> 5] = v[k];
    }
    __syncthreads();
    unsigned long long *pacc = acc + (size_t) pr * kAccWords;
    if (threadIdx.x < 4) {
        long long sum = 0;
        for (int w = 0; w < kShapePairThreads / 32; w++) sum += s_red[threadIdx.x][w];
        if (sum) atomicAdd(&pacc[threadIdx.x], (unsigned long long) sum);       // every term is >= 0
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&pacc[4], 1ull) == (unsigned long long) (split - 1);
    __syncthreads();
    if (!s_last || threadIdx.x != 0) return;
    __threadfence();
    long long tot[4];
    for (int k = 0; k < 4; k++) tot[k] = (long long) __ldcg(&pacc[k]);
    long long g, h;
    const int mir = shape_pick(tot, mirror, g, h);
    volatile ShapePairResult *o = out + pr;
    o->gap = g;
    o->he = h;
    __threadfence_system();
    o->mirrored = mir;
    for (int k = 0; k < kAccWords; k++) __stcg(&pacc[k], 0ull);
}

struct ShapeRequest : pq::Request {
    long long gap = 0, he = 0;
    int32_t mirrored = 0;
};

struct ShapeQueueDev : pq::Queue {
    uint16_t *zslice = nullptr, *grad = nullptr;   // [slots][H][W]
    uint32_t *tsig = nullptr;                      // [slots][H][bpitch]
    ShapeMaskDesc *d_descs = nullptr;              // the queue's own copy: the mask set's is reallocated by cds_shape_score_pairs
    size_t descs_cap = 0;
    ShapePairResult *h_res = nullptr, *d_res_alias = nullptr;      // pinned + mapped: the kernel writes, the dispatcher reads
    unsigned long long *d_acc = nullptr;
};

}  // namespace

struct cds_shape_pairq {
    cds_ctx *ctx = nullptr;
    const cds_shape_maskset *sms = nullptr;
    int max_batch = 64;
    int max_wait_us = 50;
    std::vector<std::unique_ptr<ShapeQueueDev>> devs;
    std::atomic<bool> stop{false};
    std::atomic<uint64_t> anon{0};
    // masks may be added to the mask set while the queue exists: a call that names a mask the queue has not seen quiesces the
    // dispatchers, refreshes the queue's descriptors and goes on
    std::atomic<int> n_masks{0};
    std::shared_mutex refresh_mu;        // a refresh takes it alone; a call that finds its mask known never touches it
};

namespace {

// the queue's descriptor copies of every mask the set holds (ctx->mu held, dispatchers idle or not started)
cds_status copy_descs(cds_shape_pairq *q)
{
    cds_ctx *ctx = q->ctx;
    for (auto &qd : q->devs) {
        const std::vector<ShapeMaskDesc> &h = q->sms->dev[qd->d].h_descs;
        cds_status st = ctx->check(cudaSetDevice(ctx->devs[qd->d].dev), "cudaSetDevice");
        if (st != CDS_OK) return st;
        if (qd->descs_cap < h.size()) {
            if (qd->d_descs) {
                st = ctx->check(cudaStreamSynchronize(qd->stream), "shape pair queue");
                if (st != CDS_OK) return st;
                cudaFree(qd->d_descs);
                qd->d_descs = nullptr; qd->descs_cap = 0;
            }
            const size_t cap = std::max<size_t>(h.size() * 2, 64);
            st = ctx->check(cudaMalloc(&qd->d_descs, cap * sizeof(ShapeMaskDesc)), "cudaMalloc(shape pair queue descriptors)");
            if (st != CDS_OK) return st;
            qd->descs_cap = cap;
        }
        if (!h.empty()) {
            st = ctx->check(cudaMemcpyAsync(qd->d_descs, h.data(), h.size() * sizeof(ShapeMaskDesc), cudaMemcpyHostToDevice, qd->stream), "descriptors H2D");
            if (st == CDS_OK) st = ctx->check(cudaStreamSynchronize(qd->stream), "descriptors H2D");
            if (st != CDS_OK) return st;
        }
    }
    q->n_masks.store(q->sms->n_masks, std::memory_order_release);
    return CDS_OK;
}

void shape_dispatcher(cds_shape_pairq *q, ShapeQueueDev *qdp)
{
    ShapeQueueDev &qd = *qdp;
    const cds_shape_maskset *sms = q->sms;
    cudaSetDevice(q->ctx->devs[qd.d].dev);
    std::vector<pq::Request *> batch;
    int last_n = 1;
    while (qd.collect(batch, q->max_batch, q->max_wait_us, last_n, q->stop)) {
        const int n = (int) batch.size();
        volatile ShapePairResult *hr = qd.h_res;
        for (int i = 0; i < n; i++) hr[i].mirrored = kResultPending;
        cudaError_t e = qd.wait_fills(batch);
        // pairs [first, first + cnt) of the batch per launch; consecutive launches share the accumulators in stream order
        for (int first = 0; first < n && e == cudaSuccess; first += kPairsPerLaunch) {
            const int cnt = std::min(kPairsPerLaunch, n - first);
            ShapePairList pl;
            for (int i = 0; i < cnt; i++) { pl.mask[i] = batch[first + i]->mask; pl.slot[i] = batch[first + i]->slot; }
            for (int i = cnt; i < kPairsPerLaunch; i++) { pl.mask[i] = 0; pl.slot[i] = 0; }
            shape_pair_batch_kernel<<<dim3((unsigned) cnt, kShapePairSplit), kShapePairThreads, 0, qd.stream>>>(
                qd.d_descs, pl, qd.zslice, qd.grad, qd.tsig, sms->W, sms->H, sms->bpitch, sms->mirror, qd.d_acc, qd.d_res_alias + first);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = qd.await_results(n, [&](int i) { return hr[i].mirrored != kResultPending; });
        qd.complete(batch, e, [&](pq::Request *r, int i) {
            ShapeRequest *sr = static_cast<ShapeRequest *>(r);
            sr->gap = hr[i].gap; sr->he = hr[i].he; sr->mirrored = hr[i].mirrored;
        });
    }
}

}  // namespace

extern "C" cds_status cds_shape_pairq_create(cds_ctx *ctx, const cds_shape_maskset *sms, int32_t max_batch, int32_t max_wait_us,
                                             int32_t cache_targets, cds_shape_pairq **out)
{
    return cds::abi_guard("cds_shape_pairq_create", [&]() -> cds_status {
        if (!ctx || !sms || !out) { set_tls_error("cds_shape_pairq_create: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        *out = nullptr;
        if (sms->ctx != ctx) return ctx->fail(CDS_ERR_BAD_ARG, "cds_shape_pairq_create: mask set belongs to another context");
        if (max_batch <= 0) max_batch = 64;
        if (max_batch > 4096) max_batch = 4096;
        if (max_wait_us < 0) max_wait_us = 0;
        std::unique_ptr<cds_shape_pairq> q(new cds_shape_pairq());
        q->ctx = ctx; q->sms = sms; q->max_batch = max_batch; q->max_wait_us = max_wait_us;
        const int W = sms->W, H = sms->H;
        const size_t px = (size_t) W * H, bytes = px * 3, bm_words = (size_t) H * sms->bpitch;
        // a lane stages target | zgap | gradient, each at a 256-byte boundary
        const size_t seg = (bytes + 255) / 256 * 256;
        const size_t stage_bytes = 2 * seg + px * sizeof(uint16_t);
        const pq::Plan plan = pq::plan(cache_targets, max_batch);
        const size_t n_slots = (size_t) plan.slots_per_queue;
        cds_status st = CDS_OK;
        for (size_t dq = 0; dq < ctx->devs.size() * (size_t) plan.queues_per_dev && st == CDS_OK; dq++) {
            const size_t d = dq / (size_t) plan.queues_per_dev;
            std::unique_ptr<ShapeQueueDev> qd(new ShapeQueueDev());
            st = ctx->check(cudaSetDevice(ctx->devs[d].dev), "cudaSetDevice");
            if (st == CDS_OK) st = qd->init(ctx, (int) d, plan.slots_per_queue, plan.lanes_per_queue, stage_bytes);
            if (st == CDS_OK) st = ctx->check(cudaMalloc(&qd->zslice, n_slots * px * sizeof(uint16_t)), "cudaMalloc(shape pair cache)");
            if (st == CDS_OK) st = ctx->check(cudaMalloc(&qd->grad, n_slots * px * sizeof(uint16_t)), "cudaMalloc(shape pair cache)");
            if (st == CDS_OK) st = ctx->check(cudaMalloc(&qd->tsig, n_slots * bm_words * sizeof(uint32_t)), "cudaMalloc(shape pair cache)");
            if (st == CDS_OK) st = ctx->check(cudaMalloc(&qd->d_acc, (size_t) kPairsPerLaunch * kAccWords * sizeof(unsigned long long)), "cudaMalloc");
            if (st == CDS_OK) st = ctx->check(cudaMemsetAsync(qd->d_acc, 0, (size_t) kPairsPerLaunch * kAccWords * sizeof(unsigned long long), qd->stream), "memset");
            if (st == CDS_OK) st = ctx->check(cudaHostAlloc(&qd->h_res, (size_t) max_batch * sizeof(ShapePairResult), cudaHostAllocMapped), "cudaHostAlloc");
            if (st == CDS_OK) st = ctx->check(cudaHostGetDevicePointer((void **) &qd->d_res_alias, qd->h_res, 0), "cudaHostGetDevicePointer");
            if (st == CDS_OK) st = ctx->check(cudaStreamSynchronize(qd->stream), "shape pair cache");
            q->devs.push_back(std::move(qd));
        }
        if (st == CDS_OK) st = copy_descs(q.get());
        if (st != CDS_OK) { cds_shape_pairq_destroy(q.release()); return st; }
        for (auto &qd : q->devs) qd->worker = std::thread(shape_dispatcher, q.get(), qd.get());
        *out = q.release();
        return CDS_OK;
    });
}

extern "C" void cds_shape_pairq_destroy(cds_shape_pairq *q)
{
    if (!q) return;
    q->stop.store(true);
    for (auto &qd : q->devs) {
        qd->stop_and_join();
        cudaSetDevice(q->ctx->devs[qd->d].dev);
        qd->release();
        for (void *p : {(void *) qd->zslice, (void *) qd->grad, (void *) qd->tsig, (void *) qd->d_descs, (void *) qd->d_acc}) if (p) cudaFree(p);
        if (qd->h_res) cudaFreeHost(qd->h_res);
    }
    cudaGetLastError();
    delete q;
}

extern "C" cds_status cds_shape_pairq_score(cds_shape_pairq *q, int32_t mask_index, uint64_t target_key,
                                            const uint8_t *target_rgb, const uint16_t *gradient, const uint8_t *zgap_rgb,
                                            int32_t target_width, int32_t target_height,
                                            int64_t *gap_out, int64_t *high_expr_out, int32_t *mirrored_out)
{
    return cds::abi_guard("cds_shape_pairq_score", [&]() -> cds_status {
        if (!q || !gap_out || !high_expr_out || !mirrored_out) { set_tls_error("cds_shape_pairq_score: NULL argument"); return CDS_ERR_BAD_ARG; }
        const cds_shape_maskset *sms = q->sms;
        if (mask_index >= q->n_masks.load(std::memory_order_acquire) && mask_index >= 0) {
            // a mask added after the queue was created: stop the dispatchers between two batches, refresh the descriptors, go on
            std::unique_lock<std::shared_mutex> rl(q->refresh_mu);
            if (mask_index >= q->n_masks.load()) {
                std::lock_guard<std::recursive_mutex> cl(q->ctx->mu);
                if (mask_index < sms->n_masks) {
                    const cds_status rs = pq::quiesced(q->devs, [&] { return copy_descs(q); });
                    if (rs != CDS_OK) return rs;
                }
            }
        }
        if (mask_index < 0 || mask_index >= q->n_masks.load(std::memory_order_acquire)) { set_tls_error("cds_shape_pairq_score: mask index out of range"); return CDS_ERR_BAD_ARG; }
        if (!gradient) { *gap_out = -1; *high_expr_out = -1; *mirrored_out = 0; return CDS_OK; }      // missing gradient supplier: Shape2DMatch...:155-158
        if (target_width != sms->W || target_height != sms->H) {
            char buf[200];
            snprintf(buf, sizeof buf, "Invalid image size - target's image size (%d, %d) must match query's image size: (%d, %d)",
                     sms->W, sms->H, target_width, target_height);
            set_tls_error(buf);
            return CDS_ERR_SIZE_MISMATCH;
        }
        if (!target_rgb) { set_tls_error("cds_shape_pairq_score: target is NULL"); return CDS_ERR_BAD_ARG; }
        const bool anonymous = target_key == 0;
        if (anonymous) target_key = 0x8000000000000000ull | ++q->anon;                    // never found again: a one-shot slot
        ShapeQueueDev &qd = *q->devs[(size_t) (target_key % q->devs.size())];
        cds_ctx *ctx = q->ctx;
        const size_t px = (size_t) sms->W * sms->H, bytes = px * 3, seg = (bytes + 255) / 256 * 256;
        ShapeRequest req;
        req.mask = mask_index;
        int lane = -1;
        cds_status st = qd.acquire(req, target_key, anonymous, lane, "cds_shape_pairq_score");
        if (st != CDS_OK) return st;
        if (lane >= 0) {
            // this thread uploads its target, zgap image and gradient through its lane and derives the slot's planes on the lane's stream
            pq::Lane &ln = qd.lanes[lane];
            const DevState &ds = ctx->devs[qd.d];
            uint8_t *h_t = ln.h_stage, *h_z = ln.h_stage + seg, *d_t = ln.d_stage, *d_z = ln.d_stage + seg;
            uint16_t *h_g = reinterpret_cast<uint16_t *>(ln.h_stage + 2 * seg);
            uint16_t *slot_grad = qd.grad + (size_t) req.slot * px;
            cudaError_t e = cudaSetDevice(ds.dev);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ln.stream);                    // the lane's previous upload has left the pinned buffer
            if (e == cudaSuccess) {
                memcpy(h_t, target_rgb, bytes);
                memcpy(h_g, gradient, px * sizeof(uint16_t));
                if (zgap_rgb) memcpy(h_z, zgap_rgb, bytes);
                e = cudaMemcpyAsync(d_t, h_t, bytes, cudaMemcpyHostToDevice, ln.stream);
            }
            if (e == cudaSuccess && zgap_rgb) e = cudaMemcpyAsync(d_z, h_z, bytes, cudaMemcpyHostToDevice, ln.stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(slot_grad, h_g, px * sizeof(uint16_t), cudaMemcpyHostToDevice, ln.stream);
            if (e == cudaSuccess) {
                launch_shape_target_planes(sms, ds, d_t, zgap_rgb ? d_z : nullptr, 1, qd.zslice + (size_t) req.slot * px,
                                           qd.tsig + (size_t) req.slot * sms->H * sms->bpitch, ln.stream);
                e = cudaGetLastError();
            }
            if (e == cudaSuccess) e = cudaEventRecord(qd.slots[req.slot].ready, ln.stream);
            st = qd.filled(req, target_key, lane, e, "cds_shape_pairq_score");
            if (st != CDS_OK) return st;
        }
        qd.wait(req);
        if (req.status != CDS_OK) { set_tls_error("cds_shape_pairq_score: the batch's kernel failed"); return req.status; }
        *gap_out = req.gap;
        *high_expr_out = req.he;
        *mirrored_out = req.mirrored;
        return CDS_OK;
    });
}

extern "C" cds_status cds_shape_pairq_get_stats(const cds_shape_pairq *q, int64_t *requests, int64_t *batches, int64_t *uploads)
{
    if (!q) { set_tls_error("cds_shape_pairq_get_stats: NULL queue"); return CDS_ERR_BAD_ARG; }
    pq::sum_stats(q->devs, requests, batches, uploads);
    return CDS_OK;
}

// Test / bench hook: drives cds_shape_pairq_score from n_threads native threads the way gradientScores' thread pool drives
// calculateMatchingScore (each thread takes the next pair of the list, blocks in the call, stores the result).  Target t is
// targets_rgb[t], gradients[t] and (zgaps_rgb == NULL: derived) zgaps_rgb[t], with key keys[t] (keys == NULL: 0, no caching).
extern "C" cds_status cds_debug_shape_pairq_drive(cds_shape_pairq *q, const uint8_t *targets_rgb, const uint16_t *gradients,
                                                  const uint8_t *zgaps_rgb, int64_t n_targets, const uint64_t *keys,
                                                  const int32_t *pair_mask, const int64_t *pair_target, int64_t n_pairs, int32_t n_threads,
                                                  int64_t *gap_out, int64_t *high_expr_out, uint8_t *mirrored_out, double *seconds_out)
{
    return cds::abi_guard("cds_debug_shape_pairq_drive", [&]() -> cds_status {
        if (!q || !targets_rgb || !gradients || !pair_mask || !pair_target || !gap_out || !high_expr_out || !seconds_out || n_threads <= 0 || n_pairs < 0) {
            set_tls_error("cds_debug_shape_pairq_drive: bad arguments");
            return CDS_ERR_BAD_ARG;
        }
        for (int64_t i = 0; i < n_pairs; i++)
            if (pair_target[i] < 0 || pair_target[i] >= n_targets) { set_tls_error("cds_debug_shape_pairq_drive: target index out of range"); return CDS_ERR_BAD_ARG; }
        const int W = q->sms->W, H = q->sms->H;
        const size_t px = (size_t) W * H;
        std::atomic<int64_t> next{0};
        std::atomic<int> failed{0};
        auto body = [&]() {
            for (;;) {
                const int64_t i = next.fetch_add(1);
                if (i >= n_pairs) return;
                int64_t gap = 0, he = 0;
                int32_t mir = 0;
                const int64_t t = pair_target[i];
                const cds_status st = cds_shape_pairq_score(q, pair_mask[i], keys ? keys[t] : 0, targets_rgb + (size_t) t * px * 3, gradients + (size_t) t * px,
                                                            zgaps_rgb ? zgaps_rgb + (size_t) t * px * 3 : nullptr, W, H, &gap, &he, &mir);
                if (st != CDS_OK) { failed.store((int) st); return; }
                gap_out[i] = gap;
                high_expr_out[i] = he;
                if (mirrored_out) mirrored_out[i] = (uint8_t) mir;
            }
        };
        const auto t0 = std::chrono::steady_clock::now();
        std::vector<std::thread> pool;
        for (int t = 0; t < n_threads; t++) pool.emplace_back(body);
        for (auto &th : pool) th.join();
        *seconds_out = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        if (failed.load()) { set_tls_error("cds_debug_shape_pairq_drive: a call failed"); return (cds_status) failed.load(); }
        return CDS_OK;
    });
}

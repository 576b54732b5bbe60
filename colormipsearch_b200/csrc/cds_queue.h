// cds_queue.h -- what the single-pair queues share: cds_pairq (pixel match, cds_pairq.cu) and cds_shape_pairq (shape score,
// cds_shape_pairq.cu).
//
// Both serve the reference's one-call-per-pair provider interface the same way.  A caller that names a target whose key is not in the
// device cache takes a free slot and an upload lane and fills the slot itself (its copies never pass through the dispatcher), leaving an
// event behind; the request then waits in a queue that one dispatcher thread drains into ONE kernel launch per batch, and every caller
// of the batch is woken by one futex broadcast.  What differs between the queues -- what a slot holds and how it is filled, the kernel
// and the result it writes -- stays with each queue: Queue below is the cache, the lanes, the request queue and the dispatcher's loop.
#pragma once

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <deque>
#include <list>
#include <memory>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <vector>

#include <climits>
#include <linux/futex.h>
#include <sys/syscall.h>
#include <unistd.h>

#include "cds_runtime.h"

namespace cds {
namespace pq {

// The pairs of a launch travel in the kernel's parameter space (no copy to enqueue) and the results are written straight into pinned
// host memory that the dispatcher polls (no copy back): a batch is one launch per kPairsPerLaunch pairs and no synchronisation.
constexpr int kPairsPerLaunch = 128;
constexpr int kIdleSpinUs = 30;          // how long an idle dispatcher polls before it goes to sleep

inline void cpu_relax()
{
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#else
    std::this_thread::yield();
#endif
}

// Callers sleep on the queue's batch counter (a futex word) instead of a condition variable: one FUTEX_WAKE releases all callers
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

// Several independent queues per device (targets are spread over them by key, each has its share of the cache, its stream and its
// dispatcher): a batch's turn-around is dominated by waking its callers and letting them back in, which costs ~1 us per caller ON
// TOP of ~35 us per batch, so several batches of a few in flight answer more calls per second than one batch of forty.
// (default: a third of the host's hardware threads, 2 .. 8 -- every queue has a dispatcher thread that polls for a moment before it
// sleeps; measured with the pixel queue on 16 cores: 40 / 80 callers reach 505 k / 660 k pairs/s with one queue, 500 k / 820 k with
// four, 520-580 k / 870-900 k with six or eight, and lose with twelve or more)
struct Plan {
    int queues_per_dev, lanes_per_queue, slots_per_queue;
};
inline Plan plan(int cache_targets, int max_batch)
{
    static const int queues_auto = (int) std::max(2u, std::min(8u, std::thread::hardware_concurrency() / 3u));
    static const int queues_per_dev = std::max(1, std::min(16, std::getenv("CDSGPU_PAIRQ_QUEUES") ? std::atoi(std::getenv("CDSGPU_PAIRQ_QUEUES")) : queues_auto));
    Plan p;
    p.queues_per_dev = queues_per_dev;
    p.lanes_per_queue = std::max(2, 8 / queues_per_dev);
    p.slots_per_queue = std::max(2 * max_batch, (cache_targets + queues_per_dev - 1) / queues_per_dev);      // a batch's slots are pinned while it runs
    return p;
}

struct Request {
    int32_t mask = 0, slot = -1;
    cudaEvent_t ready = nullptr;         // the slot's fill (nullptr: already resident)
    cds_status status = CDS_OK;
    std::atomic<bool> done{false};
};

struct CacheSlot {
    uint64_t key = 0;
    int refs = 0;                        // requests in flight that use the slot
    bool valid = false;
    bool loading = false;                // a caller is filling the slot right now
    cudaEvent_t ready = nullptr;         // recorded after the slot's fill; kept while the slot is valid
    bool ready_pending = false;          // the event may not have completed yet
    std::list<int>::iterator lru;
};

// upload staging: a device buffer + stream + pinned host buffer per lane (callers take a lane for the length of a fill)
struct Lane {
    cudaStream_t stream = nullptr;
    uint8_t *d_stage = nullptr, *h_stage = nullptr;
    bool busy = false;
};

// One dispatcher with its share of a device's cache: the slots' bookkeeping, the upload lanes, the request queue.  The slots' device
// planes and the batch buffers belong to the queue type that derives from it.
struct Queue {
    int d = 0;                           // index into ctx->devs
    cudaStream_t stream = nullptr;       // dispatcher's stream
    std::vector<CacheSlot> slots;
    std::list<int> lru;                  // least recently used first
    std::unordered_map<uint64_t, int> by_key;
    std::deque<Request *> queue;
    std::atomic<int> queued{0};          // queue.size(), readable without the mutex (the dispatcher polls it while it waits for company)
    std::atomic<bool> disp_sleeping{false};     // the dispatcher sleeps on cv_work: only then does a push pay for a notify
    std::mutex mu;
    std::condition_variable cv_work, cv_slot;
    std::atomic<uint32_t> generation{0};  // batches completed: what callers sleep on
    std::thread worker;
    bool busy = false;                   // the dispatcher is between taking a batch and finishing it
    std::condition_variable cv_idle;
    std::vector<Lane> lanes;
    int64_t batches = 0, requests = 0, uploads = 0;

    // the stream, one event per slot, the lanes with stage_bytes of staging each (the current device is d's)
    cds_status init(cds_ctx *ctx, int dev_index, int n_slots, int n_lanes, size_t stage_bytes)
    {
        d = dev_index;
        cds_status st = ctx->check(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking), "cudaStreamCreate");
        slots.resize(n_slots);
        for (int s = 0; s < n_slots && st == CDS_OK; s++) {
            st = ctx->check(cudaEventCreateWithFlags(&slots[s].ready, cudaEventDisableTiming), "cudaEventCreate");
            lru.push_back(s);
            slots[s].lru = std::prev(lru.end());
        }
        lanes.resize(n_lanes);
        for (int l = 0; l < n_lanes && st == CDS_OK; l++) {
            st = ctx->check(cudaStreamCreateWithFlags(&lanes[l].stream, cudaStreamNonBlocking), "cudaStreamCreate");
            if (st == CDS_OK) st = ctx->check(cudaMalloc(&lanes[l].d_stage, stage_bytes + 64), "cudaMalloc(pair staging)");
            if (st == CDS_OK) st = ctx->check(cudaHostAlloc(&lanes[l].h_stage, stage_bytes, cudaHostAllocDefault), "cudaHostAlloc(pair staging)");
        }
        return st;
    }

    // the dispatcher must have been joined (stop_and_join); the current device is d's
    void release()
    {
        if (stream) { cudaStreamSynchronize(stream); cudaStreamDestroy(stream); }
        for (auto &l : lanes) {
            if (l.stream) { cudaStreamSynchronize(l.stream); cudaStreamDestroy(l.stream); }
            if (l.d_stage) cudaFree(l.d_stage);
            if (l.h_stage) cudaFreeHost(l.h_stage);
        }
        for (auto &s : slots) if (s.ready) cudaEventDestroy(s.ready);
    }

    void stop_and_join()
    {
        { std::lock_guard<std::mutex> lk(mu); }
        cv_work.notify_all();
        if (worker.joinable()) worker.join();
    }

    // ---- caller side
    // Finds the key's slot or claims the least recently used free one.  lane < 0: the target is resident and the request is queued;
    // lane >= 0: the caller fills req.slot through that lane and then calls filled().
    cds_status acquire(Request &req, uint64_t key, bool anonymous, int &lane, const char *who)
    {
        lane = -1;
        std::unique_lock<std::mutex> lk(mu);
        for (;;) {
            auto it = anonymous ? by_key.end() : by_key.find(key);
            if (it != by_key.end()) {
                req.slot = it->second;
                CacheSlot &cs = slots[req.slot];
                cs.refs++;                                   // pins the slot while we wait for another caller's fill of the same target
                cv_slot.wait(lk, [&] { return !cs.loading; });
                cs.refs--;
                if (!cs.valid) { set_tls_error(std::string(who) + ": the upload of this target failed in another thread"); return CDS_ERR_CUDA; }
                if (cs.ready_pending) req.ready = cs.ready;
                break;
            }
            // a free slot (least recently used, not referenced by a request in flight) and an upload lane
            int victim = -1;
            for (int s : lru) if (slots[s].refs == 0) { victim = s; break; }
            if (victim >= 0) {
                for (size_t l = 0; l < lanes.size(); l++) if (!lanes[l].busy) { lane = (int) l; break; }
                if (lane >= 0) { req.slot = victim; break; }
            }
            // none yet: wait, then look the key up again -- another caller may have started filling this target meanwhile
            cv_slot.wait(lk);
        }
        CacheSlot &cs = slots[req.slot];
        if (lane >= 0) {
            auto old = by_key.find(cs.key);
            if (old != by_key.end() && old->second == req.slot) by_key.erase(old);
            cs.key = key; cs.valid = false; cs.loading = true;
            if (!anonymous) by_key[key] = req.slot;          // later callers with this target wait for this fill
            lanes[lane].busy = true;
            uploads++;
        }
        cs.refs++;
        lru.splice(lru.end(), lru, cs.lru);                  // most recently used (the iterator stays valid)
        if (lane < 0) push_locked(req);
        return CDS_OK;
    }

    // after the caller's fill: e = cudaSuccess when the slot's copies and kernels are enqueued and its event recorded on the lane
    cds_status filled(Request &req, uint64_t key, int lane, cudaError_t e, const char *who)
    {
        std::lock_guard<std::mutex> lk(mu);
        CacheSlot &cs = slots[req.slot];
        lanes[lane].busy = false;
        cs.loading = false;
        cds_status st = CDS_OK;
        if (e == cudaSuccess) {
            cs.valid = true; cs.ready_pending = true;
            req.ready = cs.ready;
            push_locked(req);
        } else {
            cudaGetLastError();
            st = CDS_ERR_CUDA;
            set_tls_error(std::string(who) + ": upload failed: " + cudaGetErrorString(e));
            auto mine = by_key.find(key);
            if (mine != by_key.end() && mine->second == req.slot) by_key.erase(mine);
            cs.refs--;
        }
        cv_slot.notify_all();
        return st;
    }

    // blocks until the dispatcher has answered the (queued) request
    void wait(Request &req)
    {
        if (disp_sleeping.load(std::memory_order_seq_cst)) cv_work.notify_one();
        for (;;) {
            const uint32_t g = generation.load(std::memory_order_acquire);
            if (req.done.load(std::memory_order_acquire)) break;
            futex_wait_u32(&generation, g);
        }
    }

    // ---- dispatcher side
    // The next batch (up to max_batch requests, at least one); false when the queue stops.
    bool collect(std::vector<Request *> &batch, int max_batch, int max_wait_us, int &last_n, const std::atomic<bool> &stop)
    {
        batch.clear();
        for (;;) {
            // Nothing queued: poll for a moment (the callers of the batch that has just been answered are on their way back), then
            // sleep.  Polling reads one atomic counter and takes no lock, so it does not stand in the callers' way.
            if (queued.load(std::memory_order_acquire) == 0 && !stop.load()) {
                const auto spin_until = std::chrono::steady_clock::now() + std::chrono::microseconds(kIdleSpinUs);
                while (queued.load(std::memory_order_acquire) == 0 && !stop.load() && std::chrono::steady_clock::now() < spin_until) cpu_relax();
            }
            if (queued.load(std::memory_order_acquire) == 0) {
                std::unique_lock<std::mutex> lk(mu);
                disp_sleeping.store(true, std::memory_order_seq_cst);
                cv_work.wait(lk, [&] { return stop.load() || !queue.empty(); });
                disp_sleeping.store(false, std::memory_order_seq_cst);
                if (queue.empty() && stop.load()) return false;
            }
            // wait a little for company: a batch of one costs the same launch and round trip as a batch of sixty-four
            // (as many as came last time -- the callers are a pool of threads that come back together -- or the deadline)
            const int expect = std::min(max_batch, std::max(1, last_n));
            if (queued.load(std::memory_order_acquire) < expect && max_wait_us > 0) {
                const auto deadline = std::chrono::steady_clock::now() + std::chrono::microseconds(max_wait_us);
                while (queued.load(std::memory_order_acquire) < expect && !stop.load() && std::chrono::steady_clock::now() < deadline) cpu_relax();
            }
            std::unique_lock<std::mutex> lk(mu);
            while (!queue.empty() && (int) batch.size() < max_batch) { batch.push_back(queue.front()); queue.pop_front(); }
            queued.store((int) queue.size(), std::memory_order_release);
            busy = !batch.empty();
            if (busy) break;
        }
        last_n = (int) batch.size();
        return true;
    }

    // the dispatcher's stream waits for the fills of the batch's slots
    cudaError_t wait_fills(const std::vector<Request *> &batch)
    {
        cudaError_t e = cudaSuccess;
        for (Request *r : batch)
            if (r->ready && e == cudaSuccess) e = cudaStreamWaitEvent(stream, r->ready, 0);
        return e;
    }

    // Waits for the results themselves (a microsecond after the kernel's last store) rather than for the stream: written(i) tells
    // whether result i has arrived.  Every 200 us of waiting the stream is asked whether it failed.
    template <class Written>
    cudaError_t await_results(int n, Written written)
    {
        cudaError_t e = cudaSuccess;
        auto next_query = std::chrono::steady_clock::now() + std::chrono::microseconds(200);
        for (int i = 0; i < n && e == cudaSuccess; i++) {
            while (!written(i)) {
                cpu_relax();
                if (std::chrono::steady_clock::now() >= next_query) {
                    const cudaError_t qe = cudaStreamQuery(stream);
                    if (qe == cudaSuccess) { if (!written(i)) e = cudaErrorUnknown; break; }     // finished without writing: cannot happen
                    if (qe != cudaErrorNotReady) { e = qe; break; }
                    next_query = std::chrono::steady_clock::now() + std::chrono::microseconds(200);
                }
            }
        }
        std::atomic_thread_fence(std::memory_order_acquire);
        return e;
    }

    // hands the results out (take(request, i) copies result i into the request when e == cudaSuccess) and wakes the batch's callers
    template <class Take>
    void complete(const std::vector<Request *> &batch, cudaError_t e, Take take)
    {
        const int n = (int) batch.size();
        if (e != cudaSuccess) { cudaStreamSynchronize(stream); cudaGetLastError(); }
        {
            std::lock_guard<std::mutex> lk(mu);
            batches++;
            requests += n;
            for (int i = 0; i < n; i++) {
                Request *r = batch[i];
                if (e == cudaSuccess) take(r, i);
                r->status = e == cudaSuccess ? CDS_OK : CDS_ERR_CUDA;
                CacheSlot &cs = slots[r->slot];
                cs.ready_pending = false;            // the batch ran behind the slot's event
                if (--cs.refs == 0) cv_slot.notify_all();
            }
            busy = false;
        }
        cv_idle.notify_all();
        for (int i = 0; i < n; i++) batch[i]->done.store(true, std::memory_order_release);      // (the request lives on its caller's stack: not touched after this)
        generation.fetch_add(1, std::memory_order_release);
        futex_wake_all(&generation);
    }

private:
    void push_locked(Request &req)
    {
        queue.push_back(&req);
        queued.store((int) queue.size(), std::memory_order_release);
    }
};

// Runs fn while every dispatcher of qs is between two batches and no caller can queue (a mask added after the queue was created).
template <class Q, class F>
cds_status quiesced(std::vector<std::unique_ptr<Q>> &qs, F fn)
{
    std::vector<std::unique_lock<std::mutex>> held;
    for (auto &qd : qs) {
        held.emplace_back(qd->mu);
        qd->cv_idle.wait(held.back(), [&] { return !qd->busy; });
    }
    return fn();
}

template <class Q>
void sum_stats(const std::vector<std::unique_ptr<Q>> &qs, int64_t *requests, int64_t *batches, int64_t *uploads)
{
    int64_t r = 0, b = 0, u = 0;
    for (auto &qd : qs) {
        std::lock_guard<std::mutex> lk(qd->mu);
        r += qd->requests; b += qd->batches; u += qd->uploads;
    }
    if (requests) *requests = r;
    if (batches) *batches = b;
    if (uploads) *uploads = u;
}

}  // namespace pq
}  // namespace cds

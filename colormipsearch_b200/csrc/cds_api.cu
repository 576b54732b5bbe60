// cds_api.cu -- implementation of the C ABI declared in include/cdsgpu.h: contexts, target library, mask sets and the
// pixel-match searches.  Shape scoring lives in cds_shape.cu, synthetic inputs in cds_synth.cu.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <cctype>

#include <sched.h>

#include "cds_runtime.h"
#include "cds_band.cuh"
#include "cds_cand.cuh"
#include "cds_topk.cuh"

using namespace cds;

namespace cds {
static thread_local std::string g_tls_err;
void set_tls_error(const std::string &msg) { g_tls_err = msg; }
}  // namespace cds

namespace cds {
// Most bytes a device's pool keeps for reuse (of 180 GB per B200).  The file-fed shape score works in windows of 2 048 targets
// (~20 GB of window buffers): with the earlier 8 GB limit every call paid cudaMalloc + cudaFree for the rest -- 325 instead of ~150 ms
// per 4 096 targets (bench.py shape.config2_mix.e2e_files).  An allocation that fails flushes the cache and retries (alloc below).
static constexpr size_t kPoolLimit = (size_t) 32 << 30;
static constexpr size_t kPoolBigBlock = (size_t) 256 << 20;      // blocks from this size on are cached only while ...
static constexpr size_t kPoolReserve = (size_t) 16 << 30;        // ... this much of the device is free (the current device: callers set it)

cudaError_t DevPool::alloc(void **p, size_t bytes)
{
    bytes = std::max<size_t>((bytes + 255) / 256 * 256, 256);
    auto it = free_blocks.lower_bound(bytes);
    if (it != free_blocks.end() && it->first <= std::max<size_t>(2 * bytes, (size_t) 1 << 20)) {
        *p = it->second;
        live[*p] = it->first;
        cached_bytes -= it->first;
        free_blocks.erase(it);
        return cudaSuccess;
    }
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess && !free_blocks.empty()) {      // out of memory with blocks in the cache: give them back and retry
        cudaGetLastError();
        for (auto &kv : free_blocks) cudaFree(kv.second);
        free_blocks.clear();
        cached_bytes = 0;
        e = cudaMalloc(p, bytes);
    }
    if (e == cudaSuccess) live[*p] = bytes;
    return e;
}

void DevPool::free(void *p)
{
    if (!p) return;
    auto it = live.find(p);
    if (it == live.end()) { cudaFree(p); return; }
    const size_t bytes = it->second;
    live.erase(it);
    if (cached_bytes + bytes > kPoolLimit) { cudaFree(p); return; }
    if (bytes >= kPoolBigBlock) {
        // a large block is kept only while the device has room to spare: allocations outside the pool (a library's planes, the
        // streaming buffers) do not know how to ask the pool for memory back
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) cudaGetLastError();
        else if (free_b < kPoolReserve) { cudaFree(p); return; }
    }
    free_blocks.emplace(bytes, p);
    cached_bytes += bytes;
}

void DevPool::release_all()
{
    for (auto &kv : free_blocks) cudaFree(kv.second);
    free_blocks.clear();
    cached_bytes = 0;
    for (auto &kv : live) cudaFree(kv.first);
    live.clear();
}
}  // namespace cds

cds_status cds_ctx::fail(cds_status code, const std::string &msg) const
{
    err = msg;
    set_tls_error(msg);
    return code;
}

cds_status cds_ctx::check(cudaError_t e, const char *what) const
{
    if (e == cudaSuccess) return CDS_OK;
    std::string msg = std::string(what) + ": " + cudaGetErrorString(e);
    cudaGetLastError();
    return fail(e == cudaErrorMemoryAllocation ? CDS_ERR_OOM : CDS_ERR_CUDA, msg);
}

#define CDS_TRY(expr) do { cds_status _s = (expr); if (_s != CDS_OK) return _s; } while (0)
#define CDS_CUDA(ctx, expr) CDS_TRY((ctx)->check((expr), #expr))

cds_status cds_ctx::ensure_staging(DevState &d, size_t bytes)
{
    if (d.staging_bytes >= bytes) return CDS_OK;
    CDS_CUDA(this, cudaSetDevice(d.dev));
    if (d.staging) { CDS_CUDA(this, cudaStreamSynchronize(d.stream)); cudaFree(d.staging); d.staging = nullptr; d.staging_bytes = 0; }
    CDS_CUDA(this, cudaMalloc(&d.staging, bytes + 64));
    d.staging_bytes = bytes;
    return CDS_OK;
}

cds_status cds_ctx::ensure_pinned(DevState &d, size_t bytes)
{
    if (d.h_pinned_bytes >= bytes) return CDS_OK;
    CDS_CUDA(this, cudaSetDevice(d.dev));
    if (d.h_pinned) { CDS_CUDA(this, cudaStreamSynchronize(d.stream)); cudaFreeHost(d.h_pinned); d.h_pinned = nullptr; d.h_pinned_bytes = 0; }
    CDS_CUDA(this, cudaMallocHost(&d.h_pinned, bytes));
    d.h_pinned_bytes = bytes;
    return CDS_OK;
}

cds_status cds_ctx::ensure_scratch(DevState &d, int slot, size_t bytes, void **out)
{
    if (d.scratch_bytes[slot] < bytes) {
        CDS_CUDA(this, cudaSetDevice(d.dev));
        if (d.scratch[slot]) { CDS_CUDA(this, cudaStreamSynchronize(d.stream)); cudaFree(d.scratch[slot]); d.scratch[slot] = nullptr; d.scratch_bytes[slot] = 0; }
        CDS_CUDA(this, cudaMalloc(&d.scratch[slot], bytes));
        d.scratch_bytes[slot] = bytes;
    }
    if (out) *out = d.scratch[slot];
    return CDS_OK;
}

cds_status cds_ctx::ensure_match_scratch(DevState &d)
{
    if (d.match_scratch.work_counter && d.match_scratch.acc) return CDS_OK;
    CDS_CUDA(this, cudaSetDevice(d.dev));
    if (!d.match_scratch.work_counter) CDS_CUDA(this, cudaMalloc(&d.match_scratch.work_counter, sizeof(unsigned long long)));
    if (!d.match_scratch.acc) CDS_CUDA(this, cudaMalloc(&d.match_scratch.acc, kMatchAccBytes));
    return CDS_OK;
}

cds_status cds_ctx::class_table_on(DevState &d, double tol, const cds_class_interval **out)
{
    uint64_t key;
    std::memcpy(&key, &tol, sizeof key);
    auto it = d.d_class_tabs.find(key);
    if (it != d.d_class_tabs.end()) { *out = it->second; return CDS_OK; }
    std::shared_ptr<const ClassTable> t = class_table(tol);
    if (!t) return fail(CDS_ERR_UNSUPPORTED, "match-interval table self-check failed for this zTolerance");
    cds_class_interval *dp = nullptr;
    CDS_CUDA(this, cudaSetDevice(d.dev));
    CDS_CUDA(this, cudaMalloc(&dp, t->iv.size() * sizeof(cds_class_interval)));
    CDS_CUDA(this, cudaMemcpyAsync(dp, t->iv.data(), t->iv.size() * sizeof(cds_class_interval), cudaMemcpyHostToDevice, d.stream));
    CDS_CUDA(this, cudaStreamSynchronize(d.stream));
    d.d_class_tabs[key] = dp;
    *out = dp;
    return CDS_OK;
}

// ------------------------------------------------------------------------------------------------------------------ context
extern "C" int32_t cds_abi_version(void) { return CDSGPU_ABI_VERSION; }

extern "C" const char *cds_last_error(const cds_ctx *ctx)
{
    if (ctx) {
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        g_tls_err = ctx->err;
    }
    return g_tls_err.c_str();
}

extern "C" cds_status cds_ctx_create(const int32_t *device_ids, int32_t n_dev, cds_ctx **out)
{
    return cds::abi_guard("cds_ctx_create", [&]() -> cds_status {
        if (!out) { set_tls_error("cds_ctx_create: out is NULL"); return CDS_ERR_BAD_ARG; }
        *out = nullptr;
        int visible = 0;
        cudaError_t e = cudaGetDeviceCount(&visible);
        if (e != cudaSuccess || visible == 0) {
            cudaGetLastError();
            set_tls_error(std::string("cds_ctx_create: no CUDA device (") + (e == cudaSuccess ? "0 devices" : cudaGetErrorString(e)) +
                          "); libcdsgpu has no CPU fallback");
            return CDS_ERR_NO_DEVICE;
        }
        if (n_dev < 0) { set_tls_error("cds_ctx_create: n_dev < 0"); return CDS_ERR_BAD_ARG; }
        if (n_dev == 0) { n_dev = visible; device_ids = nullptr; }
        auto ctx = new cds_ctx();
        for (int i = 0; i < n_dev; i++) {
            int id = device_ids ? device_ids[i] : i;
            if (id < 0 || id >= visible) {
                set_tls_error("cds_ctx_create: device id out of range");
                cds_ctx_destroy(ctx);
                return CDS_ERR_NO_DEVICE;
            }
            DevState d;
            d.dev = id;
            ctx->devs.push_back(d);
        }
        const RatioTable &rt = ratio_table();
        if ((int) rt.ratios.size() != CDS_NUM_RANKS) {
            set_tls_error("cds_ctx_create: ratio table self-check failed");
            cds_ctx_destroy(ctx);
            return CDS_ERR_UNSUPPORTED;
        }
        for (DevState &d : ctx->devs) {
            cds_status s = ctx->check(cudaSetDevice(d.dev), "cudaSetDevice");
            if (s == CDS_OK) s = ctx->check(cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking), "cudaStreamCreate");
            if (s == CDS_OK) {
                // the upload stream feeds the main one (file decode, inflate): its CTAs go first when an SM has room, so that the
                // latency-bound decoders stay resident next to the scoring kernels.  CDSGPU_COPY_PRIORITY=0 gives it the default priority.
                static const bool high = !(std::getenv("CDSGPU_COPY_PRIORITY") && std::atoi(std::getenv("CDSGPU_COPY_PRIORITY")) == 0);
                int lo = 0, hi = 0;
                cudaDeviceGetStreamPriorityRange(&lo, &hi);
                s = ctx->check(cudaStreamCreateWithPriority(&d.copy_stream, cudaStreamNonBlocking, high ? hi : lo), "cudaStreamCreate");
            }
            for (int i = 0; i < 2 && s == CDS_OK; i++) {
                s = ctx->check(cudaEventCreateWithFlags(&d.up_done[i], cudaEventDisableTiming), "cudaEventCreate");
                if (s == CDS_OK) s = ctx->check(cudaEventCreateWithFlags(&d.up_free[i], cudaEventDisableTiming), "cudaEventCreate");
            }
            if (s == CDS_OK) s = ctx->check(cudaEventCreate(&d.ev0), "cudaEventCreate");
            if (s == CDS_OK) s = ctx->check(cudaEventCreate(&d.ev1), "cudaEventCreate");
            if (s == CDS_OK) s = ctx->check(cudaEventCreate(&d.ev2), "cudaEventCreate");
            if (s == CDS_OK) s = ctx->check(cudaMalloc(&d.d_rank_tab, rt.rank.size() * sizeof(uint16_t)), "cudaMalloc(rank table)");
            if (s == CDS_OK) s = ctx->check(cudaMemcpy(d.d_rank_tab, rt.rank.data(), rt.rank.size() * sizeof(uint16_t), cudaMemcpyHostToDevice), "cudaMemcpy(rank table)");
            if (s != CDS_OK) { cds_ctx_destroy(ctx); return s; }
        }
        // peer access between the context's devices (mask replication); failure is not fatal
        for (DevState &a : ctx->devs)
            for (DevState &b : ctx->devs) {
                if (a.dev == b.dev) continue;
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, a.dev, b.dev) == cudaSuccess && can) {
                    cudaSetDevice(a.dev);
                    cudaDeviceEnablePeerAccess(b.dev, 0);
                    cudaGetLastError();
                }
            }
        *out = ctx;
        return CDS_OK;
    });
}

extern "C" void cds_ctx_destroy(cds_ctx *ctx)
{
    if (!ctx) return;
    for (DevState &d : ctx->devs) {
        if (cudaSetDevice(d.dev) != cudaSuccess) { cudaGetLastError(); continue; }
        if (d.stream) cudaStreamSynchronize(d.stream);
        if (d.d_rank_tab) cudaFree(d.d_rank_tab);
        for (auto &kv : d.d_class_tabs) cudaFree(kv.second);
        if (d.staging) cudaFree(d.staging);
        for (int i = 0; i < 4; i++) if (d.scratch[i]) cudaFree(d.scratch[i]);
        if (d.h_pinned) cudaFreeHost(d.h_pinned);
        if (d.pair_plane) cudaFree(d.pair_plane);
        if (d.match_scratch.work_counter) cudaFree(d.match_scratch.work_counter);
        if (d.match_scratch.acc) cudaFree(d.match_scratch.acc);
        d.pool.release_all();
        d.sb.release();
        shape_release_dev(d);
        if (d.ev0) cudaEventDestroy(d.ev0);
        if (d.ev1) cudaEventDestroy(d.ev1);
        if (d.ev2) cudaEventDestroy(d.ev2);
        for (int i = 0; i < 2; i++) {
            if (d.up_done[i]) cudaEventDestroy(d.up_done[i]);
            if (d.up_free[i]) cudaEventDestroy(d.up_free[i]);
        }
        if (d.copy_stream) cudaStreamDestroy(d.copy_stream);
        if (d.stream) cudaStreamDestroy(d.stream);
    }
    cudaGetLastError();
    delete ctx;
}

extern "C" int32_t cds_ctx_num_devices(const cds_ctx *ctx) { return ctx ? (int32_t) ctx->devs.size() : 0; }

// CPUs next to a CUDA device: /sys/bus/pci/devices/<domain:bus:device.function>/local_cpulist, e.g. "0-31,64-95"
static bool device_local_cpus(int dev, cpu_set_t &set)
{
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, dev) != cudaSuccess) { cudaGetLastError(); return false; }
    for (char *c = bus; *c; c++) *c = (char) std::tolower((unsigned char) *c);
    const std::string path = std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist";
    FILE *f = std::fopen(path.c_str(), "r");
    if (!f) return false;
    char line[1024] = {0};
    const bool got = std::fgets(line, sizeof line, f) != nullptr;
    std::fclose(f);
    if (!got) return false;
    CPU_ZERO(&set);
    int n = 0;
    for (const char *p = line; *p && *p != '\n';) {
        char *end = nullptr;
        long a = std::strtol(p, &end, 10), b = a;
        if (end == p) break;
        p = end;
        if (*p == '-') { b = std::strtol(p + 1, &end, 10); p = end; }
        for (long c = a; c <= b && c < CPU_SETSIZE; c++) { CPU_SET((int) c, &set); n++; }
        if (*p == ',') p++;
    }
    return n > 0;
}

extern "C" cds_status cds_host_alloc(cds_ctx *ctx, uint64_t bytes, void **out)
{
    return cds::abi_guard("cds_host_alloc", [&]() -> cds_status {
        if (!ctx || !out) { set_tls_error("cds_host_alloc: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        *out = nullptr;
        CDS_CUDA(ctx, cudaSetDevice(ctx->devs[0].dev));
        // Pinned pages land on the NUMA node of the allocating thread.  For the length of the allocation the thread is moved onto
        // the CPUs next to the context's first device (sysfs local_cpulist of its PCI function), so that uploads from this buffer
        // do not cross the socket interconnect; the previous affinity is restored afterwards.  Best effort: no sysfs entry, no move.
        cpu_set_t before, local;
        const bool have_before = sched_getaffinity(0, sizeof before, &before) == 0;
        const bool moved = have_before && device_local_cpus(ctx->devs[0].dev, local) && sched_setaffinity(0, sizeof local, &local) == 0;
        const cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable);
        if (moved) sched_setaffinity(0, sizeof before, &before);
        CDS_CUDA(ctx, e);
        return CDS_OK;
    });
}

extern "C" cds_status cds_host_free(cds_ctx *ctx, void *p)
{
    return cds::abi_guard("cds_host_free", [&]() -> cds_status {
        if (!ctx) { set_tls_error("cds_host_free: NULL ctx"); return CDS_ERR_BAD_ARG; }
        if (!p) return CDS_OK;
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        CDS_CUDA(ctx, cudaFreeHost(p));
        return CDS_OK;
    });
}

extern "C" cds_status cds_ctx_set_option(cds_ctx *ctx, const char *name, int64_t value)
{
    return cds::abi_guard("cds_ctx_set_option", [&]() -> cds_status {
        if (!ctx || !name) { set_tls_error("cds_ctx_set_option: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (std::strcmp(name, "match_kernel") == 0) {
            if (value < 0 || value > 3) return ctx->fail(CDS_ERR_BAD_ARG, "cds_ctx_set_option: match_kernel must be 0..3");
            ctx->match_kernel = (int) value;
            return CDS_OK;
        }
        if (std::strcmp(name, "resident_occupancy") == 0) {
            ctx->resident_occupancy = value != 0;
            return CDS_OK;
        }
        if (std::strcmp(name, "stream_chunk") == 0) {
            if (value < 1 || value > 65536) return ctx->fail(CDS_ERR_BAD_ARG, "cds_ctx_set_option: stream_chunk must be 1..65536");
            ctx->stream_chunk = value;
            return CDS_OK;
        }
        if (std::strcmp(name, "stream_chunk_bytes") == 0) {
            if (value < 1 || value > 0xC0000000ll) return ctx->fail(CDS_ERR_BAD_ARG, "cds_ctx_set_option: stream_chunk_bytes must be 1..3221225472");
            ctx->stream_chunk_bytes = value;
            return CDS_OK;
        }
        if (std::strcmp(name, "stream_chunk_tiff") == 0) {
            if (value < 1 || value > 32768) return ctx->fail(CDS_ERR_BAD_ARG, "cds_ctx_set_option: stream_chunk_tiff must be 1..32768");
            ctx->stream_chunk_tiff = value;
            return CDS_OK;
        }
        if (std::strcmp(name, "best_list_bytes") == 0) {
            if (value < 12 || value > ((int64_t) 4 << 30)) return ctx->fail(CDS_ERR_BAD_ARG, "cds_ctx_set_option: best_list_bytes must be 12..4294967296");
            ctx->best_list_bytes = value;
            return CDS_OK;
        }
        if (std::strcmp(name, "fused_ingest") == 0) { ctx->fused_ingest = value != 0; return CDS_OK; }
        if (std::strcmp(name, "cand_wait_mode") == 0) { cand_tuning().wait_mode = (int) value; return CDS_OK; }
        if (std::strcmp(name, "cand_l2_hint") == 0) { cand_tuning().l2_hint = value != 0; return CDS_OK; }
        if (std::strcmp(name, "cand_warps") == 0) { cand_tuning().warps = (int) value; return CDS_OK; }
        if (std::strcmp(name, "occupancy_kernel") == 0) { occupancy_kernel_version() = value != 0; return CDS_OK; }
        if (std::strcmp(name, "shape_inflate_window") == 0) {
            if (value < 0 || value > 8192) return ctx->fail(CDS_ERR_BAD_ARG, "cds_ctx_set_option: shape_inflate_window must be 0..8192");
            ctx->shape_inflate_window = value;
            return CDS_OK;
        }
        if (std::strcmp(name, "device_inflate") == 0) {
            if (value < 0 || value > 2) return ctx->fail(CDS_ERR_BAD_ARG, "cds_ctx_set_option: device_inflate must be 0..2");
            ctx->device_inflate = (int) value;
            return CDS_OK;
        }
        if (std::strcmp(name, "wide_lists") == 0) { ctx->wide_lists = value != 0; return CDS_OK; }
        if (std::strcmp(name, "cand_stages") == 0) { cand_tuning().stages = (int) value; return CDS_OK; }
        if (std::strcmp(name, "cand_max_rows") == 0) { cand_tuning().max_rows = (int) value; return CDS_OK; }
        return ctx->fail(CDS_ERR_BAD_ARG, std::string("cds_ctx_set_option: unknown option ") + name);
    });
}

extern "C" cds_status cds_get_last_stats(const cds_ctx *ctx, cds_search_stats *out)
{
    return cds::abi_guard("cds_get_last_stats", [&]() -> cds_status {
        if (!ctx || !out) { set_tls_error("cds_get_last_stats: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        *out = ctx->stats;
        return CDS_OK;
    });
}

// ------------------------------------------------------------------------------------------------------------------ library
namespace cds {
int choose_pitch(int W)
{
    // multiple of 4 words (16-byte rows for bulk copies), at least CDS_MIN_PAD_COLS pad words, and pitch mod 32 in
    // {8, 24} so that the same column of consecutive rows falls into different shared-memory banks
    int p = (W + CDS_MIN_PAD_COLS + 3) / 4 * 4;
    while ((p % 32) != 8 && (p % 32) != 24) p += 4;
    return p;
}
}  // namespace cds

int64_t cds_library::local_size(int dev) const
{
    // number of global indices < size that map to dev
    int D = n_dev();
    int64_t full_blocks = size / kLibBlock;
    int64_t rem = size % kLibBlock;
    int64_t blocks_on_dev = full_blocks / D + ((full_blocks % D) > dev ? 1 : 0);
    int64_t n = blocks_on_dev * kLibBlock;
    if (rem && (full_blocks % D) == dev) n += rem;
    return n;
}

cds_status cds_library::bake(int threshold)
{
    if (threshold == baked_threshold) return CDS_OK;
    for (int d = 0; d < n_dev(); d++) {
        DevState &ds = ctx->devs[d];
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        int64_t n_local = local_size(d);
        if (n_local == 0) continue;
        launch_rebake(shards[d].planes, g.total_words(n_local), threshold, ds.stream);
        ctx->stats.kernel_launches++;
        CDS_CUDA(ctx, cudaGetLastError());
    }
    for (int d = 0; d < n_dev(); d++) {
        CDS_CUDA(ctx, cudaSetDevice(ctx->devs[d].dev));
        CDS_CUDA(ctx, cudaStreamSynchronize(ctx->devs[d].stream));
    }
    baked_threshold = threshold;
    return CDS_OK;
}

cds_status cds_library::ensure_occupancy(int rings)
{
    if (occ_on_the_fly) return CDS_OK;
    if (occ_rings != rings || occ_threshold != baked_threshold) {
        for (auto &sh : shards) sh.occ_done = 0;
        occ_rings = rings;
        occ_threshold = baked_threshold;
    }
    const size_t plane_words = occupancy_target_words(g.W, g.H);
    const size_t valid_words = (size_t) g.H * CDS_NUM_SECTORS * occupancy_valid_pitch(g.W);
    const int64_t kValidChunk = 256;
    bool launched = false;
    for (int d = 0; d < n_dev(); d++) {
        Shard &sh = shards[d];
        const int64_t nl = local_size(d);
        if (sh.occ_done >= nl) continue;
        DevState &ds = ctx->devs[d];
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        if (!sh.occ) {
            cudaError_t e = cudaMalloc(&sh.occ, (size_t) sh.cap_local * plane_words * sizeof(uint32_t));
            if (e == cudaSuccess) e = cudaMalloc(&sh.valid, (size_t) std::min<int64_t>(sh.cap_local, kValidChunk) * valid_words * sizeof(uint32_t));
            if (e == cudaSuccess) e = cudaMemsetAsync(sh.occ, 0, (size_t) sh.cap_local * plane_words * sizeof(uint32_t), ds.stream);   // rows beyond the image stay clear
            if (e == cudaErrorMemoryAllocation) {
                // no room for resident bitmaps next to the code planes: searches over this library build them per target chunk
                cudaGetLastError();
                for (auto &x : shards) {
                    if (x.occ) { cudaFree(x.occ); x.occ = nullptr; }
                    if (x.valid) { cudaFree(x.valid); x.valid = nullptr; }
                    x.occ_done = 0;
                }
                occ_on_the_fly = true;
                return CDS_OK;
            }
            CDS_CUDA(ctx, e);
        }
        launch_occupancy(sh.planes, g, sh.occ_done, nl - sh.occ_done, rings, bpitch, sh.valid, std::min<int64_t>(sh.cap_local, kValidChunk), sh.occ, ds.stream,
                         false, true);
        ctx->stats.kernel_launches += 2 * ((nl - sh.occ_done + kValidChunk - 1) / kValidChunk);
        CDS_CUDA(ctx, cudaGetLastError());
        sh.occ_done = nl;
        launched = true;
    }
    if (launched)
        for (int d = 0; d < n_dev(); d++) {
            CDS_CUDA(ctx, cudaSetDevice(ctx->devs[d].dev));
            CDS_CUDA(ctx, cudaStreamSynchronize(ctx->devs[d].stream));
        }
    return CDS_OK;
}

extern "C" cds_status cds_library_create(cds_ctx *ctx, int32_t width, int32_t height, int64_t capacity, cds_library **out)
{
    return cds::abi_guard("cds_library_create", [&]() -> cds_status {
        if (!ctx || !out) { set_tls_error("cds_library_create: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        *out = nullptr;
        if (width <= 0 || height <= 0 || width > 16384 || height > 16384 || capacity <= 0)
            return ctx->fail(CDS_ERR_BAD_ARG, "cds_library_create: width/height must be in 1..16384 and capacity > 0");
        auto lib = new cds_library();
        lib->ctx = ctx;
        lib->g.W = width;
        lib->g.H = height;
        lib->g.pitch = choose_pitch(width);
        lib->g.guard = CDS_GUARD_ROWS;
        lib->bpitch = occupancy_tile_pitch(width);
        lib->capacity = capacity;
        lib->baked_threshold = 20;
        int D = (int) ctx->devs.size();
        lib->shards.resize(D);
        int64_t blocks = (capacity + kLibBlock - 1) / kLibBlock;
        int64_t blocks_per_dev = (blocks + D - 1) / D;
        for (int d = 0; d < D; d++) {
            DevState &ds = ctx->devs[d];
            cds_status s = ctx->check(cudaSetDevice(ds.dev), "cudaSetDevice");
            int64_t cap_local = blocks_per_dev * kLibBlock;
            if (cap_local > capacity && D == 1) cap_local = capacity;
            size_t words = lib->g.total_words(cap_local);
            if (s == CDS_OK) s = ctx->check(cudaMalloc(&lib->shards[d].planes, words * sizeof(uint32_t)), "cudaMalloc(library planes)");
            if (s == CDS_OK) {
                lib->shards[d].cap_local = cap_local;
                launch_fill_words(lib->shards[d].planes, words, CDS_CODE_PAD_WORD, ds.stream);
                s = ctx->check(cudaGetLastError(), "fill_words_kernel");
            }
            if (s != CDS_OK) { cds_library_destroy(lib); return s; }
        }
        for (int d = 0; d < D; d++) {
            cudaSetDevice(ctx->devs[d].dev);
            cds_status s = ctx->check(cudaStreamSynchronize(ctx->devs[d].stream), "library init");
            if (s != CDS_OK) { cds_library_destroy(lib); return s; }
        }
        *out = lib;
        return CDS_OK;
    });
}

extern "C" void cds_library_destroy(cds_library *lib)
{
    if (!lib) return;
    std::lock_guard<std::recursive_mutex> lk(lib->ctx->mu);
    for (int d = 0; d < lib->n_dev(); d++) {
        if (!lib->shards[d].planes) continue;
        cudaSetDevice(lib->ctx->devs[d].dev);
        cudaStreamSynchronize(lib->ctx->devs[d].stream);
        cudaFree(lib->shards[d].planes);
        if (lib->shards[d].occ) cudaFree(lib->shards[d].occ);
        if (lib->shards[d].valid) cudaFree(lib->shards[d].valid);
    }
    cudaGetLastError();
    delete lib;
}

extern "C" int64_t cds_library_size(const cds_library *lib) { return lib ? lib->size : 0; }

extern "C" cds_status cds_library_clear(cds_library *lib)
{
    return cds::abi_guard("cds_library_clear", [&]() -> cds_status {
        if (!lib) { set_tls_error("cds_library_clear: NULL library"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(lib->ctx->mu);
        lib->size = 0;
        for (auto &sh : lib->shards) sh.occ_done = 0;
        return CDS_OK;
    });
}

// Upload `n` RGB images that occupy consecutive global indices starting at lib->size.  `src` supplies the pixels of a run
// of images [i0, i0+cnt) (relative to the call) into a device staging pointer; used by add_rgb (H2D copy) and by the
// synthetic generator (kernel).
namespace cds {
cds_status library_append(cds_library *lib, int64_t n,
                          const std::function<cds_status(DevState &, int64_t i0, int64_t cnt, uint8_t *d_rgb)> &src,
                          int64_t *first_index)
{
    cds_ctx *ctx = lib->ctx;
    if (n < 0) return ctx->fail(CDS_ERR_BAD_ARG, "negative image count");
    if (lib->size + n > lib->capacity) return ctx->fail(CDS_ERR_CAPACITY, "library capacity exceeded");
    if (first_index) *first_index = lib->size;
    const size_t img_bytes = (size_t) lib->g.W * lib->g.H * 3;
    int64_t done = 0;
    while (done < n) {
        int64_t gidx = lib->size + done;
        int64_t in_block = kLibBlock - gidx % kLibBlock;
        int64_t cnt = std::min<int64_t>(in_block, n - done);
        int dev; int64_t local;
        lib->locate(gidx, dev, local);
        DevState &ds = ctx->devs[dev];
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        CDS_TRY(ctx->ensure_staging(ds, (size_t) kLibBlock * img_bytes));
        // the staging buffer is reused by consecutive runs on the same device: stream order keeps copy k+1 behind encode k
        CDS_TRY(src(ds, done, cnt, (uint8_t *) ds.staging));
        launch_encode_rgb((const uint8_t *) ds.staging, cnt, lib->shards[dev].planes, lib->g, local, ds.d_rank_tab,
                          lib->baked_threshold, ds.stream);
        ctx->stats.kernel_launches++;
        CDS_CUDA(ctx, cudaGetLastError());
        done += cnt;
    }
    for (DevState &ds : ctx->devs) {
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
    }
    lib->size += n;
    return CDS_OK;
}
}  // namespace cds

extern "C" cds_status cds_library_add_rgb(cds_library *lib, const uint8_t *rgb, int64_t n, int64_t *first_index)
{
    return cds::abi_guard("cds_library_add_rgb", [&]() -> cds_status {
        if (!lib) { set_tls_error("cds_library_add_rgb: NULL library"); return CDS_ERR_BAD_ARG; }
        cds_ctx *ctx = lib->ctx;
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (!rgb && n > 0) return ctx->fail(CDS_ERR_BAD_ARG, "cds_library_add_rgb: rgb is NULL");
        const size_t img_bytes = (size_t) lib->g.W * lib->g.H * 3;
        return library_append(lib, n, [&](DevState &ds, int64_t i0, int64_t cnt, uint8_t *d_rgb) -> cds_status {
            CDS_CUDA(ctx, cudaMemcpyAsync(d_rgb, rgb + (size_t) i0 * img_bytes, (size_t) cnt * img_bytes, cudaMemcpyHostToDevice, ds.stream));
            ctx->stats.h2d_bytes += (int64_t) cnt * (int64_t) img_bytes;
            return CDS_OK;
        }, first_index);
    });
}

// ------------------------------------------------------------------------------------------------------------------ mask sets
static cds_status make_shift_set(int xy_shift, int mirror, ShiftSet &out)
{
    // offsets in the order of generateShiftedMasks (API/cds/PixelMatchColorDepthSearchAlgorithm.java:113-130); duplicates of
    // (0,0) in outer rings are dropped, they cannot change a max
    out.n = 0;
    out.mirror = mirror ? 1 : 0;
    if (xy_shift < 2) { out.dx[0] = 0; out.dy[0] = 0; out.n = 1; return CDS_OK; }
    for (int i = 2; i <= xy_shift; i += 2)
        for (int xx = -i; xx <= i; xx += i)
            for (int yy = -i; yy <= i; yy += i) {
                if (i > 2 && xx == 0 && yy == 0) continue;
                if (out.n >= CDS_MAX_SHIFT_OFFSETS) return CDS_ERR_UNSUPPORTED;
                out.dx[out.n] = (int8_t) xx;
                out.dy[out.n] = (int8_t) yy;
                out.n++;
            }
    return CDS_OK;
}

extern "C" cds_status cds_maskset_create(cds_ctx *ctx, int32_t width, int32_t height, const cds_pixparams *params, cds_maskset **out)
{
    return cds::abi_guard("cds_maskset_create", [&]() -> cds_status {
        if (!ctx || !out || !params) { set_tls_error("cds_maskset_create: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        *out = nullptr;
        if (width <= 0 || height <= 0 || width > 16384 || height > 16384)
            return ctx->fail(CDS_ERR_BAD_ARG, "cds_maskset_create: width/height must be in 1..16384");
        if (params->xy_shift & 1) return ctx->fail(CDS_ERR_BAD_ARG, "XY shift parameter must be an even number.");
        if (params->xy_shift < 0) return ctx->fail(CDS_ERR_BAD_ARG, "cds_maskset_create: xy_shift < 0");
        if (params->xy_shift > CDS_MAX_XY_SHIFT) return ctx->fail(CDS_ERR_UNSUPPORTED, "cds_maskset_create: xy_shift > CDS_MAX_XY_SHIFT");
        if (params->n_rects < 0 || params->n_rects > CDS_MAX_RECTS) return ctx->fail(CDS_ERR_BAD_ARG, "cds_maskset_create: n_rects out of range");
        if (!(params->z_tolerance < 1000.0) && !std::isnan(params->z_tolerance))
            return ctx->fail(CDS_ERR_UNSUPPORTED, "cds_maskset_create: z_tolerance >= 1000 is not supported");
        auto ms = new cds_maskset();
        ms->ctx = ctx;
        ms->W = width;
        ms->H = height;
        ms->params = *params;
        if (make_shift_set(params->xy_shift, params->mirror, ms->shifts) != CDS_OK) {
            delete ms;
            return ctx->fail(CDS_ERR_UNSUPPORTED, "cds_maskset_create: too many shift offsets");
        }
        ms->rects.n = params->n_rects;
        for (int i = 0; i < params->n_rects; i++) {
            ms->rects.x0[i] = params->rects[i].x0; ms->rects.y0[i] = params->rects[i].y0;
            ms->rects.x1[i] = params->rects[i].x1; ms->rects.y1[i] = params->rects[i].y1;
        }
        ms->d_descs.assign(ctx->devs.size(), nullptr);
        ms->d_groups.assign(ctx->devs.size(), nullptr);
        ms->d_palettes.assign(ctx->devs.size(), nullptr);
        ms->d_words.assign(ctx->devs.size(), nullptr);
        ms->d_wstart.assign(ctx->devs.size(), nullptr);
        ms->store.resize(ctx->devs.size());
        // build (or fetch) the interval table now so that a bad tolerance fails here
        for (DevState &ds : ctx->devs) {
            const cds_class_interval *tab;
            cds_status s = ctx->class_table_on(ds, params->z_tolerance, &tab);
            if (s != CDS_OK) { delete ms; return s; }
        }
        *out = ms;
        return CDS_OK;
    });
}

extern "C" void cds_maskset_destroy(cds_maskset *ms)
{
    if (!ms) return;
    cds_ctx *ctx = ms->ctx;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    for (size_t d = 0; d < ctx->devs.size(); d++) {
        cudaSetDevice(ctx->devs[d].dev);
        cudaStreamSynchronize(ctx->devs[d].stream);
        if (d < ms->store.size()) {
            cds_maskset::DevStore &st = ms->store[d];
            for (cds_maskset::Arena *a : {&st.records, &st.classes, &st.crec, &st.rowstart}) ctx->devs[d].pool.free(a->p);
        }
        ctx->devs[d].pool.free(ms->d_descs[d]);
        ctx->devs[d].pool.free(ms->d_groups[d]);
        ctx->devs[d].pool.free(ms->d_palettes[d]);
        ctx->devs[d].pool.free(ms->d_words[d]);
        ctx->devs[d].pool.free(ms->d_wstart[d]);
    }
    cudaGetLastError();
    delete ms;
}

extern "C" int32_t cds_maskset_size(const cds_maskset *ms) { return ms ? (int32_t) ms->sizes.size() : 0; }

extern "C" cds_status cds_maskset_get_mask_sizes(const cds_maskset *ms, int32_t *sizes_out)
{
    return cds::abi_guard("cds_maskset_get_mask_sizes", [&]() -> cds_status {
        if (!ms || !sizes_out) { set_tls_error("cds_maskset_get_mask_sizes: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ms->ctx->mu);
        std::copy(ms->sizes.begin(), ms->sizes.end(), sizes_out);
        return CDS_OK;
    });
}

// Makes room for `used + more` bytes in a device arena; contents are preserved (device-to-device copy on growth).
static cds_status arena_reserve(cds_ctx *ctx, DevState &ds, cds_maskset::Arena &a, size_t more)
{
    if (a.used + more <= a.cap) return CDS_OK;
    size_t cap = std::max<size_t>(a.cap * 2, a.used + more);
    cap = std::max<size_t>(cap, (size_t) 1 << 20);
    void *np = nullptr;
    CDS_CUDA(ctx, ds.pool.alloc(&np, cap));
    if (a.p) {
        if (a.used) CDS_CUDA(ctx, cudaMemcpyAsync(np, a.p, a.used, cudaMemcpyDeviceToDevice, ds.stream));
        CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
        ds.pool.free(a.p);
    }
    a.p = np;
    a.cap = cap;
    return CDS_OK;
}

// Appends n masks whose RGB pixels `fill` puts into device staging memory: fill(i0, cnt, stage, stream) enqueues, on `stream`,
// whatever produces the pixels of masks [i0, i0 + cnt) of the call at `stage` (an H2D copy, or an upload of TIFF files and
// their decode).
namespace cds {
static cds_status maskset_append_body(cds_maskset *ms, int32_t n, int32_t *mask_size_out,
                                      const std::function<cds_status(int i0, int cnt, uint8_t *stage, cudaStream_t stream)> &fill);

// All or nothing: when the append fails half way (an undecodable file in a later chunk, an allocation failure), everything that
// is still in flight is drained and the mask set is rolled back to what it held before the call -- sizes, record offsets and the
// arenas of every device -- so that the next search never meets descriptors that disagree with the arenas.
cds_status maskset_append(cds_maskset *ms, int32_t n, int32_t *mask_size_out,
                          const std::function<cds_status(int i0, int cnt, uint8_t *stage, cudaStream_t stream)> &fill)
{
    cds_ctx *ctx = ms->ctx;
    const size_t first_mask = ms->sizes.size();
    const cds_maskset::DevStore &s0 = ms->store[0];
    const size_t used0[4] = {s0.records.used, s0.classes.used, s0.crec.used, s0.rowstart.used};
    const cds_status st = maskset_append_body(ms, n, mask_size_out, fill);
    if (st == CDS_OK) return CDS_OK;
    const std::string msg = ctx->err;
    for (DevState &ds : ctx->devs) {
        if (cudaSetDevice(ds.dev) != cudaSuccess) continue;
        cudaStreamSynchronize(ds.copy_stream);
        cudaStreamSynchronize(ds.stream);
    }
    cudaGetLastError();
    ms->sizes.resize(first_mask);
    ms->rec_offset.resize(first_mask);
    for (cds_maskset::DevStore &sd : ms->store) {
        sd.records.used = std::min(sd.records.used, used0[0]);
        sd.classes.used = std::min(sd.classes.used, used0[1]);
        sd.crec.used = std::min(sd.crec.used, used0[2]);
        sd.rowstart.used = std::min(sd.rowstart.used, used0[3]);
    }
    ms->descs_dirty = true;
    cudaSetDevice(ctx->devs[0].dev);
    return ctx->fail(st, msg);
}

static cds_status maskset_append_body(cds_maskset *ms, int32_t n, int32_t *mask_size_out,
                                      const std::function<cds_status(int i0, int cnt, uint8_t *stage, cudaStream_t stream)> &fill)
{
    cds_ctx *ctx = ms->ctx;
    const int D = (int) ctx->devs.size();
    const size_t img_bytes = (size_t) ms->W * ms->H * 3;
    const int H = ms->H;
    const int kChunk = maskset_append_chunk(n);     // masks per staging half: every chunk costs one host round trip (the masks' sizes)
    DevState &d0 = ctx->devs[0];
    cds_maskset::DevStore &s0 = ms->store[0];
    CDS_CUDA(ctx, cudaSetDevice(d0.dev));
    // two staging halves: the upload of chunk i+1 is queued behind the kernels of chunk i-1, not behind those of chunk i
    CDS_TRY(ctx->ensure_staging(d0, (size_t) 2 * kChunk * img_bytes));
    const cds_class_interval *class_tab;
    CDS_TRY(ctx->class_table_on(d0, ms->params.z_tolerance, &class_tab));
    CDS_TRY(ctx->ensure_scratch(d0, 1, (size_t) kChunk * sizeof(int32_t), nullptr));
    CDS_TRY(ctx->ensure_scratch(d0, 3, (size_t) kChunk * sizeof(uint64_t), nullptr));
    int32_t *d_sizes = (int32_t *) d0.scratch[1];
    uint64_t *d_off = (uint64_t *) d0.scratch[3];
    const size_t first_mask = ms->sizes.size();
    const size_t rec_used0 = s0.records.used, cls_used0 = s0.classes.used, crec_used0 = s0.crec.used, rs_used0 = s0.rowstart.used;
    CDS_TRY(arena_reserve(ctx, d0, s0.rowstart, (size_t) n * (H + 1) * sizeof(uint32_t)));
    // uploads run on the copy stream one chunk ahead of the preparation kernels (which need a host round trip per chunk)
    static const bool overlap = std::getenv("CDSGPU_MASK_OVERLAP") ? std::atoi(std::getenv("CDSGPU_MASK_OVERLAP")) != 0 : true;
    cudaStream_t up_stream = overlap ? d0.copy_stream : d0.stream;
    auto enqueue_upload = [&](int i0) -> cds_status {
        const int cnt = std::min(kChunk, n - i0);
        const int slot = (i0 / kChunk) & 1;
        uint8_t *stage = (uint8_t *) d0.staging + (size_t) slot * kChunk * img_bytes;
        if (i0 >= 2 * kChunk) CDS_CUDA(ctx, cudaStreamWaitEvent(up_stream, d0.up_free[slot], 0));
        CDS_TRY(fill(i0, cnt, stage, up_stream));
        CDS_CUDA(ctx, cudaEventRecord(d0.up_done[slot], up_stream));
        return CDS_OK;
    };
    // profiling aid (CDSGPU_MASK_TRACE=1): the host's clock at every step of the append, printed to stderr
    static const bool trace = std::getenv("CDSGPU_MASK_TRACE") != nullptr;
    const auto t_trace0 = std::chrono::steady_clock::now();
    auto tmark = [&](const char *what, int i0) {
        if (trace) std::fprintf(stderr, "# maskset_append %-28s chunk@%-5d %8.3f ms\n", what, i0, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_trace0).count());
    };
    CDS_CUDA(ctx, cudaStreamSynchronize(d0.stream));        // earlier users of the staging buffer are done
    tmark("start", 0);
    CDS_TRY(enqueue_upload(0));
    tmark("first upload enqueued", 0);
    for (int i0 = 0; i0 < n; i0 += kChunk) {
        const int cnt = std::min(kChunk, n - i0);
        const int slot = (i0 / kChunk) & 1;
        uint8_t *stage = (uint8_t *) d0.staging + (size_t) slot * kChunk * img_bytes;
        if (i0 + kChunk < n) CDS_TRY(enqueue_upload(i0 + kChunk));
        tmark("next upload enqueued", i0);
        CDS_CUDA(ctx, cudaStreamWaitEvent(d0.stream, d0.up_done[slot], 0));
        uint32_t *rowstart = (uint32_t *) ((uint8_t *) s0.rowstart.p + s0.rowstart.used);
        launch_mask_count_rows(stage, cnt, ms->W, H, ms->params.mask_threshold, ms->rects, rowstart, d0.stream);
        launch_mask_scan_rows(rowstart, cnt, H, d_sizes, d0.stream);
        ctx->stats.kernel_launches += 2;
        std::vector<int32_t> sizes(cnt);
        CDS_CUDA(ctx, cudaMemcpyAsync(sizes.data(), d_sizes, cnt * sizeof(int32_t), cudaMemcpyDeviceToHost, d0.stream));
        CDS_CUDA(ctx, cudaStreamSynchronize(d0.stream));
        tmark("sizes on the host", i0);
        std::vector<uint64_t> off(cnt);
        uint64_t total = 0;
        const uint64_t base = s0.records.used / sizeof(cds_mask_record);      // records, classes and crec advance in lock step
        for (int i = 0; i < cnt; i++) { off[i] = base + total; total += (uint64_t) sizes[i]; }
        // size the arenas once per call from the first chunk's average mask size (they still grow if the guess is short)
        uint64_t want = total;
        if (i0 == 0 && n > cnt) want = std::max<uint64_t>(total, (uint64_t) ((double) total / cnt * n * 1.15));
        CDS_TRY(arena_reserve(ctx, d0, s0.records, want * sizeof(cds_mask_record)));
        CDS_TRY(arena_reserve(ctx, d0, s0.classes, want * sizeof(uint32_t)));
        CDS_TRY(arena_reserve(ctx, d0, s0.crec, want * sizeof(uint32_t)));
        CDS_CUDA(ctx, cudaMemcpyAsync(d_off, off.data(), cnt * sizeof(uint64_t), cudaMemcpyHostToDevice, d0.stream));
        launch_mask_write_records(stage, cnt, ms->W, H, ms->params.mask_threshold, ms->rects, rowstart, d_off, d0.d_rank_tab, class_tab,
                                  (cds_mask_record *) s0.records.p, (uint32_t *) s0.classes.p, d0.stream);
        ctx->stats.kernel_launches++;
        CDS_CUDA(ctx, cudaGetLastError());
        CDS_CUDA(ctx, cudaEventRecord(d0.up_free[slot], d0.stream));        // the staging half may be overwritten
        // `off` is pageable host memory: the copy above has been staged by the time cudaMemcpyAsync returns
        s0.records.used += total * sizeof(cds_mask_record);
        s0.classes.used += total * sizeof(uint32_t);
        s0.crec.used += total * sizeof(uint32_t);
        s0.rowstart.used += (size_t) cnt * (H + 1) * sizeof(uint32_t);
        for (int i = 0; i < cnt; i++) {
            ms->sizes.push_back(sizes[i]);
            ms->rec_offset.push_back(off[i]);
            if (mask_size_out) mask_size_out[i0 + i] = sizes[i];
        }
    }
    tmark("all chunks enqueued", n);
    CDS_CUDA(ctx, cudaStreamSynchronize(d0.stream));
    tmark("records written", n);
    // replicate the new parts on the other devices
    for (int d = 1; d < D; d++) {
        DevState &dd = ctx->devs[d];
        cds_maskset::DevStore &sd = ms->store[d];
        CDS_CUDA(ctx, cudaSetDevice(dd.dev));
        struct Part { cds_maskset::Arena *dst; cds_maskset::Arena *src; size_t from; };
        const Part parts[] = {{&sd.records, &s0.records, rec_used0}, {&sd.classes, &s0.classes, cls_used0},
                              {&sd.crec, &s0.crec, crec_used0}, {&sd.rowstart, &s0.rowstart, rs_used0}};
        for (const Part &pt : parts) {
            const size_t more = pt.src->used - pt.from;
            CDS_TRY(arena_reserve(ctx, dd, *pt.dst, more));
            if (more) CDS_CUDA(ctx, cudaMemcpyPeerAsync((uint8_t *) pt.dst->p + pt.from, dd.dev, (const uint8_t *) pt.src->p + pt.from, d0.dev, more, dd.stream));
            pt.dst->used = pt.src->used;
        }
    }
    for (int d = 1; d < D; d++) {
        CDS_CUDA(ctx, cudaSetDevice(ctx->devs[d].dev));
        CDS_CUDA(ctx, cudaStreamSynchronize(ctx->devs[d].stream));
    }
    CDS_CUDA(ctx, cudaSetDevice(d0.dev));
    (void) first_mask;
    ms->descs_dirty = true;
    return CDS_OK;
}
}  // namespace cds

extern "C" cds_status cds_maskset_add_rgb(cds_maskset *ms, const uint8_t *rgb, int32_t n, int32_t *mask_size_out)
{
    return cds::abi_guard("cds_maskset_add_rgb", [&]() -> cds_status {
        if (!ms) { set_tls_error("cds_maskset_add_rgb: NULL mask set"); return CDS_ERR_BAD_ARG; }
        cds_ctx *ctx = ms->ctx;
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (n < 0 || (!rgb && n > 0)) return ctx->fail(CDS_ERR_BAD_ARG, "cds_maskset_add_rgb: bad arguments");
        if (n == 0) return CDS_OK;
        const size_t img_bytes = (size_t) ms->W * ms->H * 3;
        return maskset_append(ms, n, mask_size_out, [&](int i0, int cnt, uint8_t *stage, cudaStream_t stream) -> cds_status {
            CDS_CUDA(ctx, cudaMemcpyAsync(stage, rgb + (size_t) i0 * img_bytes, (size_t) cnt * img_bytes, cudaMemcpyHostToDevice, stream));
            ctx->stats.h2d_bytes += (int64_t) cnt * (int64_t) img_bytes;
            return CDS_OK;
        });
    });
}

cds_status cds_maskset::sync_descs()
{
    if (!descs_dirty) return CDS_OK;
    const int D = (int) ctx->devs.size();
    const int M = (int) sizes.size();
    const int n_groups = (M + CDS_PALETTE_GROUP - 1) / CDS_PALETTE_GROUP;
    std::shared_ptr<const ClassTable> ctab = class_table(params.z_tolerance);
    const bool compact_ok = ctab && ctab->max_len <= CDS_PAL_MAX_LEN && W <= 2048 && H <= 1024 && M > 0;
    n_compact_groups = 0;
    words_built = false;
    bool all_words = true;
    for (int d = 0; d < D; d++) {
        DevState &ds = ctx->devs[d];
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
        std::vector<MaskDesc> h(std::max(M, 1));
        std::vector<MaskClassRef> refs(std::max(M, 1));
        const DevStore &sd = store[d];
        for (int mi = 0; mi < M; mi++) {
            h[mi].records = (const cds_mask_record *) sd.records.p + rec_offset[mi];
            h[mi].rowstart = (const uint32_t *) sd.rowstart.p + (size_t) mi * (H + 1);
            h[mi].crec = nullptr;
            h[mi].classes = (const uint32_t *) sd.classes.p + rec_offset[mi];
            h[mi].wstart = nullptr;
            h[mi].P = sizes[mi];
            h[mi].pad = 0;
            refs[mi].classes = (const uint32_t *) sd.classes.p + rec_offset[mi];
            refs[mi].records = h[mi].records;
            refs[mi].crec = (uint32_t *) sd.crec.p + rec_offset[mi];
            refs[mi].P = sizes[mi];
            refs[mi].pad = 0;
        }
        if (d_descs[d]) { ds.pool.free(d_descs[d]); d_descs[d] = nullptr; }
        if (d_groups[d]) { ds.pool.free(d_groups[d]); d_groups[d] = nullptr; }
        if (d_palettes[d]) { ds.pool.free(d_palettes[d]); d_palettes[d] = nullptr; }
        if (d_words[d]) { ds.pool.free(d_words[d]); d_words[d] = nullptr; }
        if (d_wstart[d]) { ds.pool.free(d_wstart[d]); d_wstart[d] = nullptr; }
        std::vector<PaletteGroup> groups(std::max(n_groups, 1));
        if (d == 0) n_pal.assign(n_groups, 0);
        for (auto &g : groups) { g.palette = nullptr; g.words = nullptr; g.gstart = nullptr; g.lpal = nullptr; g.tocc = nullptr; g.n_pal = 0; g.pad = 0; }
        if (compact_ok) {
            // palettes of the compact records: mark classes per group, number them, pack intervals, rewrite records
            const size_t slots = (size_t) n_groups * (CDS_NUM_CLASSES + 1);
            MaskClassRef *d_refs = nullptr;
            uint32_t *d_flags = nullptr, *d_pidx = nullptr;
            int32_t *d_npal = nullptr;
            const cds_class_interval *class_tab = nullptr;
            cds_status st = ctx->class_table_on(ds, params.z_tolerance, &class_tab);
            if (st == CDS_OK) st = ctx->check(ds.pool.alloc((void **) &d_refs, refs.size() * sizeof(MaskClassRef)), "cudaMalloc(class refs)");
            if (st == CDS_OK) st = ctx->check(ds.pool.alloc((void **) &d_flags, slots * sizeof(uint32_t)), "cudaMalloc(palette flags)");
            if (st == CDS_OK) st = ctx->check(ds.pool.alloc((void **) &d_pidx, slots * sizeof(uint32_t)), "cudaMalloc(palette index)");
            if (st == CDS_OK) st = ctx->check(ds.pool.alloc((void **) &d_npal, n_groups * sizeof(int32_t)), "cudaMalloc(palette sizes)");
            if (st == CDS_OK) st = ctx->check(ds.pool.alloc((void **) &d_palettes[d], (size_t) n_groups * CDS_PALETTE_SIZE * sizeof(uint2)), "cudaMalloc(palettes)");
            if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(d_refs, refs.data(), refs.size() * sizeof(MaskClassRef), cudaMemcpyHostToDevice, ds.stream), "class refs H2D");
            if (st == CDS_OK) st = ctx->check(cudaMemsetAsync(d_flags, 0, slots * sizeof(uint32_t), ds.stream), "memset(palette flags)");
            std::vector<int32_t> group_pal(n_groups, 0);
            if (st == CDS_OK) {
                launch_palette_mark(d_refs, M, d_flags, ds.stream);
                launch_palette_scan(d_flags, n_groups, d_pidx, d_npal, ds.stream);
                launch_palette_fill(d_flags, d_pidx, n_groups, class_tab, d_palettes[d], ds.stream);
                launch_palette_records(d_refs, M, d_pidx, d_npal, ds.stream);
                ctx->stats.kernel_launches += 4;
                st = ctx->check(cudaGetLastError(), "palette kernels");
            }
            if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(group_pal.data(), d_npal, n_groups * sizeof(int32_t), cudaMemcpyDeviceToHost, ds.stream), "palette sizes D2H");
            if (st == CDS_OK) st = ctx->check(cudaStreamSynchronize(ds.stream), "palette build");
            ds.pool.free(d_refs);
            ds.pool.free(d_flags);
            ds.pool.free(d_pidx);
            ds.pool.free(d_npal);
            if (st != CDS_OK) return st;
            int compact = 0;
            for (int g = 0; g < n_groups; g++) {
                if (group_pal[g] >= CDS_PALETTE_SIZE) continue;   // a staged palette keeps one entry for idle lanes
                groups[g].palette = d_palettes[d] + (size_t) g * CDS_PALETTE_SIZE;
                groups[g].n_pal = group_pal[g];
                if (d == 0) n_pal[g] = group_pal[g];
                compact++;
                for (int m = g * CDS_PALETTE_GROUP; m < std::min(M, (g + 1) * CDS_PALETTE_GROUP); m++) h[m].crec = refs[m].crec;
            }
            n_compact_groups = compact;
        }
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_descs[d], h.size() * sizeof(MaskDesc)));
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_groups[d], groups.size() * sizeof(PaletteGroup)));
        CDS_CUDA(ctx, cudaMemcpyAsync(d_descs[d], h.data(), h.size() * sizeof(MaskDesc), cudaMemcpyHostToDevice, ds.stream));
        // word lists of the candidate kernel (cds_cand.cuh): per-(mask, row) counts, per-(group, row) runs, row starts, fill.
        // They reference the groups' palettes; when a group has more classes than a palette holds, the lists of the whole set
        // carry the packed intervals instead (WIDE, 32 instead of 16 bits per mask pixel and list).
        const bool words_ok = M > 0 && W <= 2048 && H <= 1024 && (params.xy_shift == 0 || params.xy_shift == 2 || params.xy_shift == 4) &&
                              compact_ok;
        const bool wide = words_ok && (n_compact_groups != n_groups || ctx->wide_lists);
        if (d == 0) wide_lpal = wide;
        if (words_ok) {
            uint32_t *d_grow = nullptr;
            const int HT = occupancy_tile_rows(H);              // the lists are ordered by rows of 8 x 4 tiles
            const size_t gs_n = (size_t) n_groups * (HT + 1), ms_n = (size_t) M * (HT + 1);
            const cds_class_interval *class_tab = nullptr;
            cds_status st = ctx->class_table_on(ds, params.z_tolerance, &class_tab);
            // d_wstart: per-mask entry offsets [M][H+1], per-mask bit offsets [M][H+1], entry row starts [G][H+1], bit row starts [G][H+1]
            if (st == CDS_OK) st = ctx->check(ds.pool.alloc((void **) &d_wstart[d], (2 * ms_n + 2 * gs_n) * sizeof(uint32_t)), "cudaMalloc(word row starts)");
            if (st == CDS_OK) st = ctx->check(ds.pool.alloc((void **) &d_grow, 2 * gs_n * sizeof(uint32_t)), "cudaMalloc(group rows)");
            if (st == CDS_OK) st = ctx->check(cudaMemsetAsync(d_grow, 0, 2 * gs_n * sizeof(uint32_t), ds.stream), "memset(group rows)");
            std::vector<uint32_t> grow(2 * gs_n, 0);
            uint32_t *d_wcount = d_wstart[d], *d_bcount = d_wstart[d] + ms_n;
            if (st == CDS_OK) {
                launch_words_count(d_descs[d], M, W, H, params.mirror != 0, class_tab, d_wcount, d_bcount, ds.stream);
                launch_words_group_rows(d_wcount, M, HT, d_grow, ds.stream);
                launch_words_group_rows(d_bcount, M, HT, d_grow + gs_n, ds.stream);
                ctx->stats.kernel_launches += 3;
                st = ctx->check(cudaGetLastError(), "word count kernels");
            }
            if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(grow.data(), d_grow, 2 * gs_n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ds.stream), "group rows D2H");
            if (st == CDS_OK) st = ctx->check(cudaStreamSynchronize(ds.stream), "word count");
            ds.pool.free(d_grow);
            if (st != CDS_OK) return st;
            uint64_t total[2] = {0, 0};
            for (int a = 0; a < 2; a++)
                for (int g = 0; g < n_groups; g++) {
                    uint32_t *row = grow.data() + a * gs_n + (size_t) g * (HT + 1);
                    for (int y = 0; y < HT; y++) { const uint32_t c = row[y]; row[y] = (uint32_t) total[a]; total[a] += c; }
                    row[HT] = (uint32_t) total[a];
                }
            if (total[0] < ((uint64_t) 1 << 32) && total[1] < ((uint64_t) 1 << 32)) {
                uint32_t *d_gstart = d_wstart[d] + 2 * ms_n, *d_bstart = d_gstart + gs_n;
                // d_words: the entries, then the palette references
                // d_words: the entries, the ticket bounds, then the palette references
                const size_t n_tocc = words_tocc_count((uint32_t) total[0]);
                CDS_CUDA(ctx, ds.pool.alloc((void **) &d_words[d], std::max<uint64_t>(total[0], 1) * sizeof(uint4) + n_tocc * sizeof(uint32_t) +
                                                                       std::max<uint64_t>(total[1], 1) * (wide ? sizeof(uint32_t) : sizeof(uint16_t))));
                uint4 *d_entries = reinterpret_cast<uint4 *>(d_words[d]);
                uint32_t *d_tocc = reinterpret_cast<uint32_t *>(d_entries + std::max<uint64_t>(total[0], 1));
                uint16_t *d_lpal = reinterpret_cast<uint16_t *>(d_tocc + n_tocc);
                CDS_CUDA(ctx, cudaMemcpyAsync(d_gstart, grow.data(), 2 * gs_n * sizeof(uint32_t), cudaMemcpyHostToDevice, ds.stream));
                for (int m = 0; m < M; m++) h[m].wstart = d_wcount + (size_t) m * (HT + 1);
                for (int g = 0; g < n_groups; g++) {
                    groups[g].words = d_entries;
                    groups[g].gstart = d_gstart + (size_t) g * (HT + 1);
                    groups[g].lpal = d_lpal;
                    groups[g].tocc = d_tocc;
                }
                CDS_CUDA(ctx, cudaMemcpyAsync(d_descs[d], h.data(), h.size() * sizeof(MaskDesc), cudaMemcpyHostToDevice, ds.stream));
                launch_words_fill(d_descs[d], M, W, H, params.mirror != 0, class_tab, d_gstart, d_bstart, d_bcount, d_entries, d_lpal, ds.stream, wide);
                ctx->stats.kernel_launches++;
                CDS_CUDA(ctx, cudaGetLastError());
                {
                    // bucket order inside every tile row (cds_cand.cuh): sort into a scratch copy, copy back
                    uint4 *d_sorted = nullptr;
                    uint32_t *d_tables = nullptr;
                    const size_t tbl = (size_t) 2 * n_groups * words_bucket_count(W, H) * sizeof(uint32_t);
                    cds_status st2 = ctx->check(ds.pool.alloc((void **) &d_sorted, std::max<uint64_t>(total[0], 1) * sizeof(uint4)), "cudaMalloc(sorted words)");
                    if (st2 == CDS_OK) st2 = ctx->check(ds.pool.alloc((void **) &d_tables, tbl), "cudaMalloc(bucket tables)");
                    if (st2 == CDS_OK) {
                        launch_words_bucket_sort(d_entries, d_gstart, n_groups, W, H, d_tables, d_sorted, ds.stream);
                        ctx->stats.kernel_launches += 3;
                        st2 = ctx->check(cudaGetLastError(), "bucket sort kernels");
                    }
                    if (st2 == CDS_OK) st2 = ctx->check(cudaMemcpyAsync(d_entries, d_sorted, total[0] * sizeof(uint4), cudaMemcpyDeviceToDevice, ds.stream), "sorted words copy");
                    if (st2 == CDS_OK) {
                        launch_words_tocc(d_entries, (uint32_t) total[0], d_tocc, ds.stream);
                        ctx->stats.kernel_launches++;
                        st2 = ctx->check(cudaGetLastError(), "ticket bounds kernel");
                    }
                    cudaStreamSynchronize(ds.stream);
                    ds.pool.free(d_sorted);
                    ds.pool.free(d_tables);
                    if (st2 != CDS_OK) return st2;
                }
                CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));      // `grow` is pageable memory
            } else {
                all_words = false;
            }
        } else {
            all_words = false;
        }
        CDS_CUDA(ctx, cudaMemcpyAsync(d_groups[d], groups.data(), groups.size() * sizeof(PaletteGroup), cudaMemcpyHostToDevice, ds.stream));
        CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
    }
    words_built = all_words;
    descs_dirty = false;
    return CDS_OK;
}

// ------------------------------------------------------------------------------------------------------------------ searches
namespace cds {
cds_status launch_match_view(cds_ctx *ctx, const cds_maskset *ms, const TargetView &tv, int d, int m0, int mc, int32_t *d_scores,
                             cudaStream_t stream, cudaEvent_t ev0, cudaEvent_t ev1)
{
    const int choice = ctx->match_kernel;      // 0 = automatic, 1 = candidate, 2 = band, 3 = gather (cds_ctx_set_option)
    const bool batched_ok = mc >= band_min_masks() && tv.occ_ready && (m0 % CDS_PALETTE_GROUP) == 0;
    const bool cand_ok = batched_ok && (choice == 0 || choice == 1) && ms->d_words[d] && ms->words_built && cand_kernel_supported(ms->params.xy_shift, tv.g);
    const bool band_ok = batched_ok && choice != 3 && band_kernel_supported(ms->params.xy_shift, tv.g);
    if (cand_ok || band_ok) CDS_TRY(ctx->ensure_match_scratch(ctx->devs[d]));
    const MatchScratch &scratch = ctx->devs[d].match_scratch;
    if (ev0) cudaEventRecord(ev0, stream);
    if (cand_ok) {
        // the largest palette of the launch's groups, plus its idle entry: what the kernel stages
        int pal_entries = 0;
        for (int g = m0 / CDS_PALETTE_GROUP; g <= (m0 + mc - 1) / CDS_PALETTE_GROUP; g++) pal_entries = std::max(pal_entries, ms->n_pal[g] + 1);
        int launches = launch_pixelmatch_cand(ms->d_descs[d] + m0, mc, tv.planes, tv.g, tv.n, tv.occ, tv.bpitch,
                                              ms->d_groups[d] + m0 / CDS_PALETTE_GROUP, ms->params.xy_shift, ms->params.mirror != 0,
                                              d_scores, scratch, stream, ms->wide_lpal, tv.bands, pal_entries);
        ctx->stats.kernel_launches += launches;
        ctx->stats.match_kernel_launches += launches;
        ctx->stats.match_kernel = 1;
    } else if (band_ok) {
        int launches = launch_pixelmatch_band(ms->d_descs[d] + m0, mc, tv.planes, tv.g, tv.n, tv.occ, tv.bpitch,
                                              ms->d_groups[d] + m0 / CDS_PALETTE_GROUP, ms->params.xy_shift, ms->params.mirror != 0,
                                              d_scores, scratch, stream);
        ctx->stats.kernel_launches += launches;
        ctx->stats.match_kernel_launches += launches;
        ctx->stats.match_kernel = 2;
    } else {
        launch_pixelmatch_gather(ms->d_descs[d] + m0, mc, tv.planes, tv.g, tv.n, ms->shifts, d_scores, stream);
        int launches = (mc + 32767) / 32768;
        ctx->stats.kernel_launches += launches;
        ctx->stats.match_kernel_launches += launches;
        ctx->stats.match_kernel = 3;
    }
    if (ev1) cudaEventRecord(ev1, stream);
    return ctx->check(cudaGetLastError(), "pixel match kernel");
}

bool batched_kernel_supported(int xy_shift, const PlaneGeom &g)
{
    return cand_kernel_supported(xy_shift, g) || band_kernel_supported(xy_shift, g);
}
}  // namespace cds

extern "C" cds_status cds_debug_cand_config(int32_t width, int32_t height, int32_t xy_shift, int32_t palette_entries, int32_t wide,
                                            int32_t *warps, int32_t *rows_per_band, int32_t *stages, int64_t *smem_bytes)
{
    return cds::abi_guard("cds_debug_cand_config", [&]() -> cds_status {
        if (width <= 0 || height <= 0 || width > 2048 || height > 1024 || !(xy_shift == 0 || xy_shift == 2 || xy_shift == 4) ||
            palette_entries < 1 || palette_entries > CDS_PALETTE_SIZE || !warps || !rows_per_band || !stages || !smem_bytes) {
            set_tls_error("cds_debug_cand_config: bad argument");
            return CDS_ERR_BAD_ARG;
        }
        PlaneGeom g;
        g.W = width; g.H = height; g.pitch = choose_pitch(width); g.guard = CDS_GUARD_ROWS;
        const CandShape c = cand_launch_shape(xy_shift, g, wide ? 0 : palette_entries);
        *warps = c.ok ? c.warps : 0;
        *rows_per_band = c.ok ? c.rows_per_band : 0;
        *stages = c.ok ? c.n_stages : 0;
        *smem_bytes = c.ok ? (int64_t) c.smem_bytes : 0;
        return CDS_OK;
    });
}

extern "C" cds_status cds_debug_library_bands(cds_library *lib, int32_t data_threshold, int32_t xy_shift, uint8_t *bands_out)
{
    return cds::abi_guard("cds_debug_library_bands", [&]() -> cds_status {
        if (!lib) { set_tls_error("cds_debug_library_bands: NULL library"); return CDS_ERR_BAD_ARG; }
        cds_ctx *ctx = lib->ctx;
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (data_threshold < 0 || data_threshold > 255 || !(xy_shift == 0 || xy_shift == 2 || xy_shift == 4))
            return ctx->fail(CDS_ERR_BAD_ARG, "cds_debug_library_bands: bad data_threshold or xy_shift");
        if (lib->size == 0) return CDS_OK;
        if (!bands_out) return ctx->fail(CDS_ERR_BAD_ARG, "cds_debug_library_bands: NULL output");
        CDS_TRY(lib->bake(data_threshold));
        CDS_TRY(lib->ensure_occupancy(xy_shift / 2));
        if (lib->occ_on_the_fly) return ctx->fail(CDS_ERR_UNSUPPORTED, "cds_debug_library_bands: the library builds its occupancy per chunk");
        const int tp = lib->bpitch, HT = occupancy_tile_rows(lib->g.H), row_bytes = CDS_NUM_SECTORS * tp;
        for (int64_t gi = 0; gi < lib->size; gi++) {
            int d = 0;
            int64_t t = 0;
            lib->locate(gi, d, t);
            DevState &ds = ctx->devs[d];
            CDS_CUDA(ctx, cudaSetDevice(ds.dev));
            const uint32_t *src = lib->shards[d].occ + (size_t) t * occupancy_target_words(lib->g.W, lib->g.H) + occupancy_band_offset(tp);
            CDS_CUDA(ctx, cudaMemcpy2D(bands_out + (size_t) gi * HT * row_bytes, (size_t) row_bytes, src, (size_t) occupancy_row_pitch(tp) * 4,
                                       (size_t) row_bytes, (size_t) HT, cudaMemcpyDeviceToHost));
        }
        return CDS_OK;
    });
}

namespace {

// Runs the match kernel of one device for masks [m0, m0+mc) against the device's local targets [0, n_local):
// d_scores[(m - m0) * n_local + t] = score word.
cds_status launch_match(cds_ctx *ctx, const cds_maskset *ms, cds_library *lib, int d, int m0, int mc, int64_t n_local,
                        int32_t *d_scores)
{
    DevState &ds = ctx->devs[d];
    TargetView tv;
    tv.planes = lib->shards[d].planes;
    tv.occ = lib->shards[d].occ;
    tv.g = lib->g;
    tv.bpitch = lib->bpitch;
    tv.n = n_local;
    tv.occ_ready = lib->shards[d].occ && lib->shards[d].occ_done >= n_local && lib->occ_rings == ms->params.xy_shift / 2 &&
                   lib->occ_threshold == lib->baked_threshold;
    tv.bands = tv.occ_ready;
    return launch_match_view(ctx, ms, tv, d, m0, mc, d_scores, ds.stream, ds.ev0, ds.ev1);
}

cds_status check_search_args(cds_ctx *ctx, const cds_maskset *ms, const cds_library *lib)
{
    if (ms->ctx != ctx || lib->ctx != ctx) return ctx->fail(CDS_ERR_BAD_ARG, "mask set / library belong to another context");
    if (ms->W != lib->g.W || ms->H != lib->g.H) {
        char buf[200];
        snprintf(buf, sizeof buf, "Invalid image size - target's image size (%d, %d) must match query's image size: (%d, %d)",
                 ms->W, ms->H, lib->g.W, lib->g.H);
        return ctx->fail(CDS_ERR_SIZE_MISMATCH, buf);
    }
    return CDS_OK;
}

void reset_stats(cds_ctx *ctx)
{
    ctx->stats = cds_search_stats{};
}

}  // namespace

extern "C" cds_status cds_search_dense(cds_ctx *ctx, const cds_maskset *ms_c, cds_library *lib, int32_t *scores, uint8_t *mirrored)
{
    return cds::abi_guard("cds_search_dense", [&]() -> cds_status {
        if (!ctx || !ms_c || !lib) { set_tls_error("cds_search_dense: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        cds_maskset *ms = const_cast<cds_maskset *>(ms_c);
        CDS_TRY(check_search_args(ctx, ms, lib));
        const int M = (int) ms->sizes.size();
        const int64_t T = lib->size;
        if (M == 0 || T == 0) return CDS_OK;
        if (!scores) return ctx->fail(CDS_ERR_BAD_ARG, "cds_search_dense: scores is NULL");
        reset_stats(ctx);
        CDS_TRY(ms->sync_descs());
        CDS_TRY(lib->bake(ms->params.data_threshold));
        if (batched_kernel_supported(ms->params.xy_shift, lib->g) && M >= band_min_masks()) CDS_TRY(lib->ensure_occupancy(ms->params.xy_shift / 2));
        const int D = lib->n_dev();
        // mask chunking bounds the per-device score buffer to ~256 MiB
        std::vector<int32_t *> d_scores(D, nullptr);
        cds_status st = CDS_OK;
        int64_t max_local = 0;
        for (int d = 0; d < D; d++) max_local = std::max(max_local, lib->local_size(d));
        int mchunk = (int) std::max<int64_t>(1, std::min<int64_t>(M, ((int64_t) 64 << 20) / std::max<int64_t>(max_local, 1)));
        if (mchunk < M && mchunk > CDS_PALETTE_GROUP) mchunk -= mchunk % CDS_PALETTE_GROUP;   // keep chunks aligned to palette groups
        for (int d = 0; d < D && st == CDS_OK; d++) {
            st = ctx->check(cudaSetDevice(ctx->devs[d].dev), "cudaSetDevice");
            if (st == CDS_OK) st = ctx->ensure_scratch(ctx->devs[d], 0, (size_t) mchunk * std::max<int64_t>(lib->local_size(d), 1) * sizeof(int32_t), (void **) &d_scores[d]);
            if (st == CDS_OK) st = ctx->ensure_pinned(ctx->devs[d], (size_t) mchunk * std::max<int64_t>(lib->local_size(d), 1) * sizeof(int32_t));
        }
        double match_ms = 0;
        for (int m0 = 0; m0 < M && st == CDS_OK; m0 += mchunk) {
            const int mc = std::min(mchunk, M - m0);
            for (int d = 0; d < D && st == CDS_OK; d++) {
                const int64_t nl = lib->local_size(d);
                if (nl == 0) continue;
                DevState &ds = ctx->devs[d];
                st = ctx->check(cudaSetDevice(ds.dev), "cudaSetDevice");
                if (st == CDS_OK) st = launch_match(ctx, ms, lib, d, m0, mc, nl, d_scores[d]);
                if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(ds.h_pinned, d_scores[d], (size_t) mc * nl * sizeof(int32_t), cudaMemcpyDeviceToHost, ds.stream), "scores D2H");
                ctx->stats.d2h_bytes += (int64_t) mc * nl * (int64_t) sizeof(int32_t);
            }
            double chunk_ms = 0;
            for (int d = 0; d < D && st == CDS_OK; d++) {
                const int64_t nl = lib->local_size(d);
                if (nl == 0) continue;
                DevState &ds = ctx->devs[d];
                cudaSetDevice(ds.dev);
                st = ctx->check(cudaStreamSynchronize(ds.stream), "pixel match");
                if (st != CDS_OK) break;
                float ms_f = 0;
                cudaEventElapsedTime(&ms_f, ds.ev0, ds.ev1);
                chunk_ms = std::max(chunk_ms, (double) ms_f);
                const int32_t *h = (const int32_t *) ds.h_pinned;
                for (int mi = 0; mi < mc; mi++)
                    for (int64_t l = 0; l < nl; l++) {
                        int32_t w = h[(size_t) mi * nl + l];
                        size_t o = (size_t) (m0 + mi) * T + lib->global_of(d, l);
                        scores[o] = w & ~CDS_SCORE_MIRROR_BIT;
                        if (mirrored) mirrored[o] = (w & CDS_SCORE_MIRROR_BIT) ? 1 : 0;
                    }
            }
            match_ms += chunk_ms;
        }
        ctx->stats.match_kernel_ms = match_ms;
        ctx->stats.total_device_ms = match_ms;
        ctx->stats.comparisons = (int64_t) M * T;
        return st;
    });
}

// smallest score s in [1, P] with ColorMIPSearch.isMatch true (API/cds/ColorMIPSearch.java:42-45); P+1 when none.
namespace cds {
int32_t min_matching_score(int32_t P, double pct_positive_pixels)
{
    if (P <= 0) return 1;   // empty mask scores 0 and never matches (score > 0 fails)
    const double thr = pct_positive_pixels / 100;
    auto ok = [&](int32_t s) { return s > 0 && (double) (float) ((double) s / (double) P) > thr; };
    if (!ok(P)) return P + 1;
    int32_t a = 1, b = P;    // invariant: ok(b)
    while (a < b) { int32_t mid = a + (b - a) / 2; if (ok(mid)) b = mid; else a = mid + 1; }
    return b;
}
}  // namespace cds

extern "C" cds_status cds_search_topk(cds_ctx *ctx, const cds_maskset *ms_c, cds_library *lib, int32_t k, double pct_positive_pixels,
                                      int32_t *out_score, int64_t *out_target, uint8_t *out_mirrored, int32_t *out_count)
{
    return cds::abi_guard("cds_search_topk", [&]() -> cds_status {
        if (!ctx || !ms_c || !lib) { set_tls_error("cds_search_topk: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        cds_maskset *ms = const_cast<cds_maskset *>(ms_c);
        CDS_TRY(check_search_args(ctx, ms, lib));
        if (k <= 0 || k > topk_max_k()) return ctx->fail(CDS_ERR_BAD_ARG, "cds_search_topk: k must be in 1..4096");
        const int M = (int) ms->sizes.size();
        const int64_t T = lib->size;
        if (M == 0) return CDS_OK;
        if (!out_score || !out_target || !out_count) return ctx->fail(CDS_ERR_BAD_ARG, "cds_search_topk: NULL output");
        reset_stats(ctx);
        for (int m = 0; m < M; m++) out_count[m] = 0;
        if (T == 0) return CDS_OK;
        CDS_TRY(ms->sync_descs());
        CDS_TRY(lib->bake(ms->params.data_threshold));
        const bool batched = batched_kernel_supported(ms->params.xy_shift, lib->g) && M >= band_min_masks();
        if (batched && ctx->resident_occupancy) CDS_TRY(lib->ensure_occupancy(ms->params.xy_shift / 2));
        if (batched && (lib->occ_on_the_fly || !ctx->resident_occupancy))
            return search_library_chunked(ctx, ms, lib, k, pct_positive_pixels, out_score, out_target, out_mirrored, out_count);
        const int D = lib->n_dev();
        std::vector<int32_t> min_score(M);
        for (int m = 0; m < M; m++) min_score[m] = min_matching_score(ms->sizes[m], pct_positive_pixels);

        int64_t max_local = 0;
        for (int d = 0; d < D; d++) max_local = std::max(max_local, lib->local_size(d));
        int mchunk = (int) std::max<int64_t>(1, std::min<int64_t>(M, ((int64_t) 512 << 20) / std::max<int64_t>(max_local, 1)));
        if (mchunk < M && mchunk > CDS_PALETTE_GROUP) mchunk -= mchunk % CDS_PALETTE_GROUP;   // keep chunks aligned to palette groups
        std::vector<int32_t *> d_scores(D, nullptr);
        std::vector<int32_t *> d_min(D, nullptr);
        std::vector<uint64_t *> d_keys(D, nullptr);
        std::vector<int32_t *> d_counts(D, nullptr);
        cds_status st = CDS_OK;
        const size_t keys_bytes = (size_t) M * k * sizeof(uint64_t);
        for (int d = 0; d < D && st == CDS_OK; d++) {
            DevState &ds = ctx->devs[d];
            st = ctx->check(cudaSetDevice(ds.dev), "cudaSetDevice");
            if (st == CDS_OK) st = ctx->ensure_scratch(ds, 0, (size_t) mchunk * std::max<int64_t>(lib->local_size(d), 1) * sizeof(int32_t), (void **) &d_scores[d]);
            if (st == CDS_OK) st = ctx->ensure_scratch(ds, 1, M * sizeof(int32_t), (void **) &d_min[d]);
            if (st == CDS_OK) st = ctx->ensure_scratch(ds, 2, keys_bytes, (void **) &d_keys[d]);
            if (st == CDS_OK) st = ctx->ensure_scratch(ds, 3, M * sizeof(int32_t), (void **) &d_counts[d]);
            if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(d_min[d], min_score.data(), M * sizeof(int32_t), cudaMemcpyHostToDevice, ds.stream), "min scores H2D");
            if (st == CDS_OK) st = ctx->check(cudaMemsetAsync(d_counts[d], 0, M * sizeof(int32_t), ds.stream), "memset");
            if (st == CDS_OK) st = ctx->ensure_pinned(ds, keys_bytes + M * sizeof(int32_t));
        }
        double match_ms = 0, total_ms = 0;
        for (int m0 = 0; m0 < M && st == CDS_OK; m0 += mchunk) {
            const int mc = std::min(mchunk, M - m0);
            for (int d = 0; d < D && st == CDS_OK; d++) {
                const int64_t nl = lib->local_size(d);
                if (nl == 0) continue;
                DevState &ds = ctx->devs[d];
                st = ctx->check(cudaSetDevice(ds.dev), "cudaSetDevice");
                if (st == CDS_OK) st = launch_match(ctx, ms, lib, d, m0, mc, nl, d_scores[d]);
                if (st == CDS_OK) {
                    launch_topk(d_scores[d], mc, nl, d_min[d] + m0, k, 0, d_keys[d] + (size_t) m0 * k, d_counts[d] + m0, ds.stream);
                    ctx->stats.kernel_launches++;
                    cudaEventRecord(ds.ev2, ds.stream);
                    st = ctx->check(cudaGetLastError(), "topk kernel");
                }
            }
            double chunk_ms = 0, chunk_total_ms = 0;
            for (int d = 0; d < D && st == CDS_OK; d++) {
                if (lib->local_size(d) == 0) continue;
                DevState &ds = ctx->devs[d];
                cudaSetDevice(ds.dev);
                st = ctx->check(cudaStreamSynchronize(ds.stream), "pixel match + topk");
                if (st != CDS_OK) break;
                float ms_f = 0;
                cudaEventElapsedTime(&ms_f, ds.ev0, ds.ev1);
                chunk_ms = std::max(chunk_ms, (double) ms_f);
                cudaEventElapsedTime(&ms_f, ds.ev0, ds.ev2);
                chunk_total_ms = std::max(chunk_total_ms, (double) ms_f);
            }
            match_ms += chunk_ms;
            total_ms += chunk_total_ms;
        }
        // read back per-device lists and merge on the host (no collective: nothing is reduced across devices)
        std::vector<std::vector<uint64_t>> h_keys(D);
        std::vector<std::vector<int32_t>> h_counts(D);
        for (int d = 0; d < D && st == CDS_OK; d++) {
            if (lib->local_size(d) == 0) continue;
            DevState &ds = ctx->devs[d];
            cudaSetDevice(ds.dev);
            uint8_t *hp = (uint8_t *) ds.h_pinned;
            st = ctx->check(cudaMemcpyAsync(hp, d_keys[d], keys_bytes, cudaMemcpyDeviceToHost, ds.stream), "keys D2H");
            if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(hp + keys_bytes, d_counts[d], M * sizeof(int32_t), cudaMemcpyDeviceToHost, ds.stream), "counts D2H");
            ctx->stats.d2h_bytes += (int64_t) keys_bytes + (int64_t) M * 4;
        }
        for (int d = 0; d < D && st == CDS_OK; d++) {
            if (lib->local_size(d) == 0) continue;
            DevState &ds = ctx->devs[d];
            cudaSetDevice(ds.dev);
            st = ctx->check(cudaStreamSynchronize(ds.stream), "topk D2H");
            if (st != CDS_OK) break;
            const uint8_t *hp = (const uint8_t *) ds.h_pinned;
            h_keys[d].assign((const uint64_t *) hp, (const uint64_t *) hp + (size_t) M * k);
            h_counts[d].assign((const int32_t *) (hp + keys_bytes), (const int32_t *) (hp + keys_bytes) + M);
        }
        if (st == CDS_OK) {
            struct Item { int32_t score; int64_t target; uint8_t mir; };
            std::vector<Item> items;
            for (int m = 0; m < M; m++) {
                items.clear();
                for (int d = 0; d < D; d++) {
                    if (h_counts[d].empty()) continue;
                    int c = std::min(h_counts[d][m], k);
                    for (int i = 0; i < c; i++) {
                        uint64_t key = h_keys[d][(size_t) m * k + i];
                        Item it;
                        topk_decode_key(key, it.score, it.target, it.mir);
                        it.target = lib->global_of(d, it.target);
                        items.push_back(it);
                    }
                }
                std::sort(items.begin(), items.end(), [](const Item &a, const Item &b) {
                    if (a.score != b.score) return a.score > b.score;
                    return a.target < b.target;
                });
                int c = (int) std::min<size_t>(items.size(), (size_t) k);
                out_count[m] = c;
                for (int i = 0; i < c; i++) {
                    out_score[(size_t) m * k + i] = items[i].score;
                    out_target[(size_t) m * k + i] = items[i].target;
                    if (out_mirrored) out_mirrored[(size_t) m * k + i] = items[i].mir;
                }
            }
        }
        ctx->stats.match_kernel_ms = match_ms;
        ctx->stats.total_device_ms = total_ms;
        ctx->stats.comparisons = (int64_t) M * T;
        return st;
    });
}

extern "C" cds_status cds_score_pair_rgb(cds_ctx *ctx, const cds_maskset *ms, int32_t mask_index, const uint8_t *target_rgb,
                                         int32_t target_width, int32_t target_height,
                                         int32_t *score_out, double *ratio_out, int32_t *mirrored_out)
{
    return cds::abi_guard("cds_score_pair_rgb", [&]() -> cds_status {
        if (!ctx || !ms || !score_out || !ratio_out || !mirrored_out) { set_tls_error("cds_score_pair_rgb: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (mask_index < 0 || mask_index >= (int) ms->sizes.size()) return ctx->fail(CDS_ERR_BAD_ARG, "cds_score_pair_rgb: mask index out of range");
        const int P = ms->sizes[mask_index];
        if (P == 0) { *score_out = 0; *ratio_out = 0; *mirrored_out = 0; return CDS_OK; }   // PixelMatch...:169-170 (before the size check)
        if (target_width != ms->W || target_height != ms->H) {
            char buf[200];
            snprintf(buf, sizeof buf, "Invalid image size - target's image size (%d, %d) must match query's image size: (%d, %d)",
                     ms->W, ms->H, target_width, target_height);
            return ctx->fail(CDS_ERR_SIZE_MISMATCH, buf);
        }
        if (!target_rgb) return ctx->fail(CDS_ERR_BAD_ARG, "cds_score_pair_rgb: target is NULL");
        // a one-slot library on device 0, kept between calls (this is the call the reference's thread pool makes per pair)
        cds_ctx *c = ctx;
        cds_maskset *msm = const_cast<cds_maskset *>(ms);
        CDS_TRY(msm->sync_descs());
        DevState &d0 = c->devs[0];
        CDS_CUDA(c, cudaSetDevice(d0.dev));
        PlaneGeom g;
        g.W = ms->W; g.H = ms->H; g.pitch = choose_pitch(ms->W); g.guard = CDS_GUARD_ROWS;
        const size_t words = g.total_words(1);
        const size_t img_bytes = (size_t) g.W * g.H * 3;
        CDS_TRY(c->ensure_staging(d0, (size_t) kLibBlock * img_bytes));
        if (d0.pair_W != g.W || d0.pair_H != g.H) {
            if (d0.pair_plane) { CDS_CUDA(c, cudaStreamSynchronize(d0.stream)); cudaFree(d0.pair_plane); d0.pair_plane = nullptr; }
            CDS_CUDA(c, cudaMalloc(&d0.pair_plane, words * sizeof(uint32_t) + sizeof(int32_t)));
            launch_fill_words(d0.pair_plane, words, CDS_CODE_PAD_WORD, d0.stream);     // guard rows / pad columns stay pad words
            d0.pair_W = g.W; d0.pair_H = g.H;
        }
        uint32_t *plane = d0.pair_plane;
        int32_t *d_score = (int32_t *) (plane + words);
        cds_status st = c->check(cudaMemcpyAsync(d0.staging, target_rgb, img_bytes, cudaMemcpyHostToDevice, d0.stream), "pair H2D");
        if (st == CDS_OK) {
            launch_encode_rgb((const uint8_t *) d0.staging, 1, plane, g, 0, d0.d_rank_tab, ms->params.data_threshold, d0.stream);
            launch_pixelmatch_gather(msm->d_descs[0] + mask_index, 1, plane, g, 1, ms->shifts, d_score, d0.stream);
            st = c->check(cudaGetLastError(), "pair kernels");
        }
        int32_t w = 0;
        if (st == CDS_OK) st = c->check(cudaMemcpyAsync(&w, d_score, sizeof w, cudaMemcpyDeviceToHost, d0.stream), "pair D2H");
        if (st == CDS_OK) st = c->check(cudaStreamSynchronize(d0.stream), "pair sync");
        if (st != CDS_OK) return st;
        *score_out = w & ~CDS_SCORE_MIRROR_BIT;
        *mirrored_out = (w & CDS_SCORE_MIRROR_BIT) ? 1 : 0;
        *ratio_out = (double) *score_out / (double) P;     // :194
        return CDS_OK;
    });
}

// ------------------------------------------------------------------------------------------------------------------ post-processing
extern "C" int64_t cds_shape_score_2d(int64_t gradient_area_gap, int64_t high_expression_area)
{
    // GradientAreaGapUtils.calculate2DShapeScore, API/cds/GradientAreaGapUtils.java:199-207
    if (gradient_area_gap >= 0 && high_expression_area >= 0) return gradient_area_gap + high_expression_area / 3;
    return -1;
}

extern "C" double cds_normalized_score(int32_t pixel_match_score, int64_t shape_score, int64_t max_pixel_match, int64_t max_shape_score)
{
    // GradientAreaGapUtils.calculateNormalizedScore, API/cds/GradientAreaGapUtils.java:219-235
    if (pixel_match_score == 0 || max_pixel_match == 0 || shape_score < 0 || max_shape_score <= 0) return pixel_match_score;
    double normalized_pixel_score = (double) pixel_match_score / (double) max_pixel_match;
    double normalized_shape_score = (double) shape_score / (double) max_shape_score;
    double bounded = std::fmin(std::fmax(normalized_shape_score * 2.5, 0.002), 1.);
    return normalized_pixel_score / bounded * 100;
}

extern "C" cds_status cds_normalize_scores(const int32_t *pixel_scores, const int64_t *gaps, const int64_t *high_exprs, int64_t n,
                                           float *normalized_out)
{
    return cds::abi_guard("cds_normalize_scores", [&]() -> cds_status {
        // CalculateGradientScoresCmd.normalizeScores, TOOLS/CalculateGradientScoresCmd.java:616-645: the maxima run over the
        // mask's matches, the normalised score is stored as float
        if (n < 0 || (n > 0 && (!pixel_scores || !gaps || !high_exprs || !normalized_out))) {
            set_tls_error("cds_normalize_scores: bad arguments");
            return CDS_ERR_BAD_ARG;
        }
        int64_t max_pix = 0, max_shape = -1;
        bool any = false;
        for (int64_t i = 0; i < n; i++) {
            max_pix = std::max<int64_t>(max_pix, pixel_scores[i]);
            int64_t s = cds_shape_score_2d(gaps[i], high_exprs[i]);
            if (!any || s > max_shape) { max_shape = s; any = true; }
        }
        for (int64_t i = 0; i < n; i++) {
            int64_t s = cds_shape_score_2d(gaps[i], high_exprs[i]);
            normalized_out[i] = (float) cds_normalized_score(pixel_scores[i], s, max_pix, max_shape);
        }
        return CDS_OK;
    });
}

// ------------------------------------------------------------------------------------------------------------------ test hooks
extern "C" cds_status cds_debug_encode_colors(cds_ctx *ctx, const uint8_t *rgb, int64_t n, int32_t data_threshold, uint32_t *codes_out)
{
    return cds::abi_guard("cds_debug_encode_colors", [&]() -> cds_status {
        if (!ctx || (n > 0 && (!rgb || !codes_out))) { set_tls_error("cds_debug_encode_colors: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (n <= 0) return CDS_OK;
        DevState &d0 = ctx->devs[0];
        CDS_CUDA(ctx, cudaSetDevice(d0.dev));
        uint8_t *d_rgb = nullptr;
        uint32_t *d_codes = nullptr;
        cds_status st = ctx->check(cudaMalloc(&d_rgb, (size_t) n * 3), "cudaMalloc");
        if (st == CDS_OK) st = ctx->check(cudaMalloc(&d_codes, (size_t) n * 4), "cudaMalloc");
        if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(d_rgb, rgb, (size_t) n * 3, cudaMemcpyHostToDevice, d0.stream), "H2D");
        if (st == CDS_OK) {
            launch_encode_colors(d_rgb, n, d0.d_rank_tab, data_threshold, d_codes, d0.stream);
            st = ctx->check(cudaGetLastError(), "encode_colors_kernel");
        }
        if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(codes_out, d_codes, (size_t) n * 4, cudaMemcpyDeviceToHost, d0.stream), "D2H");
        if (st == CDS_OK) st = ctx->check(cudaStreamSynchronize(d0.stream), "sync");
        if (d_rgb) cudaFree(d_rgb);
        if (d_codes) cudaFree(d_codes);
        return st;
    });
}

extern "C" cds_status cds_debug_class_intervals(double z_tolerance, int32_t sector, int32_t rank,
                                                uint32_t *lo1, uint32_t *len1, uint32_t *lo2, uint32_t *len2)
{
    return cds::abi_guard("cds_debug_class_intervals", [&]() -> cds_status {
        if (sector < 0 || sector >= CDS_NUM_SECTORS || rank < 0 || rank >= CDS_NUM_RANKS || !lo1 || !len1 || !lo2 || !len2) {
            set_tls_error("cds_debug_class_intervals: bad arguments");
            return CDS_ERR_BAD_ARG;
        }
        cds_class_interval iv = class_interval(z_tolerance, sector, rank);
        *lo1 = iv.lo1; *len1 = iv.len1; *lo2 = iv.lo2; *len2 = iv.len2;
        return CDS_OK;
    });
}

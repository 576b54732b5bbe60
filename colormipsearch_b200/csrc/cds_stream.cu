// cds_stream.cu -- cds_search_stream_rgb: the batched seam of the reference,
// ColorMIPSearchProcessor.findAllColorDepthMatches(masks, targets)
// (colormipsearch-tools/src/main/java/org/janelia/colormipsearch/cmd/cdsprocess/ColorMIPSearchProcessor.java:8-12,
//  LocalColorMIPSearchProcessor.java:55-116), for targets that live in HOST memory and need not stay on the device.
//
// Targets are cut into chunks; chunk c goes to device c mod D.  Per device two streams: the copy stream uploads chunk i+1
// into the other half of a double-buffered staging area while the compute stream encodes chunk i into code planes, builds
// its occupancy bitmap, runs the match kernel for ALL masks against it, selects the chunk's per-mask top-K and folds it into
// the running per-mask lists.  The host only enqueues; it blocks once, at the end, to read the lists back and merge them
// over the devices.  With pinned host memory the call runs at the rate of the slower of PCIe and the match kernel.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>

#include "cds_runtime.h"
#include "cds_band.cuh"
#include "cds_bestsel.cuh"
#include "cds_topk.cuh"
#include "cds_tiff.h"

using namespace cds;

#define CDS_TRY(expr) do { cds_status _s = (expr); if (_s != CDS_OK) return _s; } while (0)
#define CDS_CUDA(ctx, expr) CDS_TRY((ctx)->check((expr), #expr))

void cds::StreamBufs::release()
{
    for (int i = 0; i < 2; i++) {
        if (staging[i]) cudaFree(staging[i]);
        if (h2d_done[i]) cudaEventDestroy(h2d_done[i]);
        if (enc_done[i]) cudaEventDestroy(enc_done[i]);
        staging[i] = nullptr; h2d_done[i] = nullptr; enc_done[i] = nullptr;
    }
    void *bufs[] = {planes, occ, valid, scores, keys_chunk, keys_run, counts_chunk, counts_run, min_score, strip_counter};
    for (void *b : bufs) if (b) cudaFree(b);
    strip_counter = nullptr;
    planes = occ = valid = nullptr; scores = nullptr; keys_chunk = keys_run = nullptr;
    counts_chunk = counts_run = min_score = nullptr;
    for (int i = 0; i < 2; i++) {
        if (comp[i]) cudaFree(comp[i]);
        if (d_strips[i]) cudaFree(d_strips[i]);
        if (h_strips[i]) cudaFreeHost(h_strips[i]);
        comp[i] = nullptr; d_strips[i] = nullptr; h_strips[i] = nullptr;
    }
    comp_cap = strips_cap = 0;
    for (cudaEvent_t e : timing) cudaEventDestroy(e);
    timing.clear();
    if (copy_stream) cudaStreamDestroy(copy_stream);
    copy_stream = nullptr;
    W = H = 0; chunk = 0; m_cap = 0; key_cap = 0;
}

namespace {

cds_status ensure_stream_bufs(cds_ctx *ctx, DevState &ds, const PlaneGeom &g, int bpitch, int64_t chunk, int64_t M, int64_t k, bool upload,
                              int staging_slots)
{
    StreamBufs &sb = ds.sb;
    CDS_CUDA(ctx, cudaSetDevice(ds.dev));
    if (!sb.copy_stream) {
        CDS_CUDA(ctx, cudaStreamCreateWithFlags(&sb.copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CDS_CUDA(ctx, cudaEventCreateWithFlags(&sb.h2d_done[i], cudaEventDisableTiming));
            CDS_CUDA(ctx, cudaEventCreateWithFlags(&sb.enc_done[i], cudaEventDisableTiming));
        }
    }
    const size_t img_bytes = (size_t) g.W * g.H * 3;
    if (sb.W != g.W || sb.H != g.H || sb.chunk < chunk) {
        CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
        CDS_CUDA(ctx, cudaStreamSynchronize(sb.copy_stream));
        for (int i = 0; i < 2; i++) if (sb.staging[i]) { cudaFree(sb.staging[i]); sb.staging[i] = nullptr; sb.staging_cap[i] = 0; }
        if (sb.planes) { cudaFree(sb.planes); sb.planes = nullptr; }
        if (sb.occ) { cudaFree(sb.occ); sb.occ = nullptr; }
        if (sb.valid) { cudaFree(sb.valid); sb.valid = nullptr; }
        if (sb.scores) { cudaFree(sb.scores); sb.scores = nullptr; }
        sb.chunk = 0; sb.m_cap = 0;
        const size_t words = g.total_words(chunk);
        const size_t bm_words = (size_t) chunk * occupancy_target_words(g.W, g.H);
        const size_t valid_words = (size_t) chunk * g.H * CDS_NUM_SECTORS * occupancy_valid_pitch(g.W);
        (void) words; (void) bpitch;
        CDS_CUDA(ctx, cudaMalloc(&sb.occ, bm_words * sizeof(uint32_t)));
        CDS_CUDA(ctx, cudaMalloc(&sb.valid, valid_words * sizeof(uint32_t)));
        CDS_CUDA(ctx, cudaMemsetAsync(sb.occ, 0, bm_words * sizeof(uint32_t), ds.stream));      // rows beyond the image stay clear
        sb.W = g.W; sb.H = g.H; sb.chunk = chunk;
    }
    if (upload && !sb.planes) {
        // code planes of one chunk: only searches over host targets need them
        const size_t words = g.total_words(sb.chunk);
        CDS_CUDA(ctx, cudaMalloc(&sb.planes, words * sizeof(uint32_t)));
        launch_fill_words(sb.planes, words, CDS_CODE_PAD_WORD, ds.stream);      // guard rows stay pad words for ever
        CDS_CUDA(ctx, cudaGetLastError());
    }
    // RGB staging: two halves for uploaded pixels, one for the two-kernel TIFF path, none for the fused TIFF ingest
    for (int i = 0; i < staging_slots; i++) {
        const size_t need = (size_t) chunk * img_bytes + 64;
        if (sb.staging_cap[i] >= need) continue;
        CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
        CDS_CUDA(ctx, cudaStreamSynchronize(sb.copy_stream));
        if (sb.staging[i]) { cudaFree(sb.staging[i]); sb.staging[i] = nullptr; sb.staging_cap[i] = 0; }
        CDS_CUDA(ctx, cudaMalloc(&sb.staging[i], need));
        sb.staging_cap[i] = need;
    }
    if (sb.m_cap < M) {
        CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
        if (sb.scores) cudaFree(sb.scores);
        if (sb.counts_chunk) cudaFree(sb.counts_chunk);
        if (sb.counts_run) cudaFree(sb.counts_run);
        if (sb.min_score) cudaFree(sb.min_score);
        sb.scores = nullptr; sb.counts_chunk = sb.counts_run = sb.min_score = nullptr; sb.m_cap = 0;
        CDS_CUDA(ctx, cudaMalloc(&sb.scores, (size_t) M * sb.chunk * sizeof(int32_t)));
        CDS_CUDA(ctx, cudaMalloc(&sb.counts_chunk, (size_t) M * sizeof(int32_t)));
        CDS_CUDA(ctx, cudaMalloc(&sb.counts_run, (size_t) M * sizeof(int32_t)));
        CDS_CUDA(ctx, cudaMalloc(&sb.min_score, (size_t) M * sizeof(int32_t)));
        sb.m_cap = M;
    }
    if (sb.key_cap < M * k) {
        CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
        if (sb.keys_chunk) cudaFree(sb.keys_chunk);
        if (sb.keys_run) cudaFree(sb.keys_run);
        sb.keys_chunk = sb.keys_run = nullptr; sb.key_cap = 0;
        CDS_CUDA(ctx, cudaMalloc(&sb.keys_chunk, (size_t) M * k * sizeof(uint64_t)));
        CDS_CUDA(ctx, cudaMalloc(&sb.keys_run, (size_t) M * k * sizeof(uint64_t)));
        sb.key_cap = M * k;
    }
    return CDS_OK;
}

// staging of the TIFF source: both streams are drained before anything is replaced
cds_status ensure_tiff_bufs(cds_ctx *ctx, DevState &ds, size_t comp_bytes, size_t n_strips)
{
    StreamBufs &sb = ds.sb;
    CDS_CUDA(ctx, cudaSetDevice(ds.dev));
    if (!sb.strip_counter) CDS_CUDA(ctx, cudaMalloc(&sb.strip_counter, 64));
    if (sb.comp_cap >= comp_bytes && sb.strips_cap >= n_strips) return CDS_OK;
    CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
    CDS_CUDA(ctx, cudaStreamSynchronize(sb.copy_stream));
    if (sb.comp_cap < comp_bytes) {
        for (int i = 0; i < 2; i++) {
            if (sb.comp[i]) { cudaFree(sb.comp[i]); sb.comp[i] = nullptr; }
            CDS_CUDA(ctx, cudaMalloc(&sb.comp[i], comp_bytes));
        }
        sb.comp_cap = comp_bytes;
    }
    if (sb.strips_cap < n_strips) {
        const size_t cap = std::max(n_strips, sb.strips_cap * 2);
        for (int i = 0; i < 2; i++) {
            if (sb.d_strips[i]) { cudaFree(sb.d_strips[i]); sb.d_strips[i] = nullptr; }
            if (sb.h_strips[i]) { cudaFreeHost(sb.h_strips[i]); sb.h_strips[i] = nullptr; }
            CDS_CUDA(ctx, cudaMalloc(&sb.d_strips[i], cap * sizeof(TiffStrip)));
            CDS_CUDA(ctx, cudaMallocHost(&sb.h_strips[i], cap * sizeof(TiffStrip)));
        }
        sb.strips_cap = cap;
    }
    return CDS_OK;
}

}  // namespace

namespace cds {

// The chunk plan of a search over host targets: (device, first target, count), chunks dealt round-robin over the devices.  Pixels
// (offsets == nullptr): equal chunks.  TIFF files: the first chunks of every device are short (256, 512, ...) so that the match kernel
// starts early -- a full chunk needs milliseconds of parsing, upload and ingest before its first comparison -- and what is left after
// the ramp is cut into equal chunks (a short last chunk would leave most SMs idle during its match kernel: the kernel hands out whole
// targets).  A chunk of files also ends where its bytes would exceed `byte_cap` (what the strip table addresses with 32 bits).
std::vector<StreamChunk> stream_chunk_plan(int D, int64_t n_targets, int64_t chunk, const int64_t *offsets, uint64_t byte_cap)
{
    std::vector<StreamChunk> plan;
    if (D < 1 || chunk < 1) return plan;
    int64_t f = 0;
    int64_t even = 0;                      // chunk length after the ramp (0: not there yet)
    for (int64_t c = 0; f < n_targets; c++) {
        int64_t want = chunk;
        if (offsets) {
            const int64_t ramp = (int64_t) 256 << std::min<int64_t>(c / D, 8);
            if (ramp < chunk) {
                want = ramp;
            } else {
                if (even == 0) {
                    const int64_t rest = n_targets - f, per_round = chunk * D;
                    const int64_t rounds = (rest + per_round - 1) / per_round;
                    even = std::max<int64_t>(1, (rest + rounds * D - 1) / (rounds * D));
                }
                want = std::min(chunk, even);
            }
        }
        int64_t cnt = std::min<int64_t>(want, n_targets - f);
        if (offsets)
            while (cnt > 1 && (uint64_t) (offsets[f + cnt] - offsets[f]) > byte_cap) cnt = (cnt + 1) / 2;
        plan.push_back({(int) (c % D), f, cnt});
        f += cnt;
    }
    return plan;
}

}  // namespace cds

// Test hook: the plan above, without a device.
extern "C" cds_status cds_debug_stream_plan(int32_t n_devices, int64_t n_targets, int64_t chunk, const int64_t *offsets, int64_t byte_cap,
                                            int64_t capacity, int32_t *dev_out, int64_t *first_out, int64_t *count_out, int64_t *n_out)
{
    return cds::abi_guard("cds_debug_stream_plan", [&]() -> cds_status {
        if (!n_out || n_devices < 1 || chunk < 1 || n_targets < 0 || byte_cap < 1 || capacity < 0) { set_tls_error("cds_debug_stream_plan: bad argument"); return CDS_ERR_BAD_ARG; }
        const std::vector<cds::StreamChunk> plan = cds::stream_chunk_plan(n_devices, n_targets, chunk, offsets, (uint64_t) byte_cap);
        *n_out = (int64_t) plan.size();
        if ((int64_t) plan.size() > capacity) { set_tls_error("cds_debug_stream_plan: capacity too small"); return CDS_ERR_CAPACITY; }
        for (size_t i = 0; i < plan.size(); i++) {
            if (dev_out) dev_out[i] = plan[i].d;
            if (first_out) first_out[i] = plan[i].first;
            if (count_out) count_out[i] = plan[i].cnt;
        }
        return CDS_OK;
    });
}

namespace {

// targets given as TIFF files stored back to back (cds_search_stream_tiff)
struct TiffSource {
    const uint8_t *blob;
    const int64_t *offsets;
};

// `all` selects the second mode of the streaming search: instead of per-mask top-K lists, every pair that passes isMatch.
struct AllMatchesOut {
    int64_t capacity;
    int32_t *mask;
    int64_t *target;
    int32_t *score;
    uint8_t *mirrored;
    int64_t *count;
};

// The third mode: the passing pairs stay on the devices (within "best_list_bytes" per device) and only the best-matches selection
// over them (csrc/cds_bestsel.cu) comes back.
struct BestMatchesOut {
    const cds_target_groups *groups;
    int32_t top_lines, top_samples_per_line, top_matches_per_sample;
    int64_t capacity;
    int32_t *mask;
    int64_t *target;
    int32_t *score;
    uint8_t *mirrored;
    int64_t *count;
};

cds_status stream_search_impl(cds_ctx *ctx, const cds_maskset *ms_c, const uint8_t *targets_rgb, int64_t n_targets,
                              int32_t k, double pct_positive_pixels,
                              int32_t *out_score, int64_t *out_target, uint8_t *out_mirrored, int32_t *out_count, const AllMatchesOut *all,
                              cds_library *resident, const TiffSource *tiff = nullptr, const BestMatchesOut *best = nullptr)
{
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    cds_maskset *ms = const_cast<cds_maskset *>(ms_c);
    if (ms->ctx != ctx) return ctx->fail(CDS_ERR_BAD_ARG, "mask set belongs to another context");
    const bool collect = all || best;      // every passing pair goes to a device list
    if (!collect && (k <= 0 || k > topk_max_k())) return ctx->fail(CDS_ERR_BAD_ARG, "cds_search_stream_rgb: k must be in 1..4096");
    if (collect) k = 1;
    if (resident) n_targets = resident->size;
    if (!resident && !tiff && (n_targets < 0 || (n_targets > 0 && !targets_rgb))) return ctx->fail(CDS_ERR_BAD_ARG, "cds_search_stream_rgb: bad target array");
    if (tiff && (n_targets < 0 || (n_targets > 0 && (!tiff->blob || !tiff->offsets)))) return ctx->fail(CDS_ERR_BAD_ARG, "cds_search_stream_tiff: bad target array");
    const int M = (int) ms->sizes.size();
    if (all) {
        if (!all->count || all->capacity < 0 || (all->capacity > 0 && (!all->mask || !all->target || !all->score)))
            return ctx->fail(CDS_ERR_BAD_ARG, "cds_search_stream_matches_rgb: bad output arrays");
        *all->count = 0;
    }
    if (best) {
        if (!best->count || best->capacity < 0 || (best->capacity > 0 && (!best->mask || !best->target || !best->score)))
            return ctx->fail(CDS_ERR_BAD_ARG, "best matches: bad output arrays");
        *best->count = 0;
    }
    if (M == 0) return CDS_OK;
    if (!collect && (!out_score || !out_target || !out_count)) return ctx->fail(CDS_ERR_BAD_ARG, "cds_search_stream_rgb: NULL output");
    ctx->stats = cds_search_stats{};
    if (!collect) for (int m = 0; m < M; m++) out_count[m] = 0;
    if (n_targets == 0) return CDS_OK;
    // A mask set that has changed since its last search still needs its palettes and word lists (sync_descs: a few small kernels and
    // several host round trips, ~3 ms for 1 000 masks).  The search over files does not wait for that: the first chunk's upload, ingest
    // and occupancy rows are put on the copy stream first and run while the lists are built; its match kernel waits for both.
    bool descs_pending = tiff != nullptr && ms->descs_dirty;
    if (!descs_pending) CDS_TRY(ms->sync_descs());

    const int D = (int) ctx->devs.size();
    PlaneGeom g;
    g.W = ms->W; g.H = ms->H; g.pitch = choose_pitch(ms->W); g.guard = CDS_GUARD_ROWS;
    const int bpitch = occupancy_tile_pitch(g.W);
    const size_t img_bytes = (size_t) g.W * g.H * 3;
    if (resident) {
        if (resident->ctx != ctx) return ctx->fail(CDS_ERR_BAD_ARG, "library belongs to another context");
        g = resident->g;
        CDS_TRY(resident->bake(ms->params.data_threshold));
    }
    const bool fused_ingest = ctx->fused_ingest != 0 && g.W <= 2048;      // the fused kernel marks 32-pixel chunks in a 64-bit mask
    int64_t chunk = std::min<int64_t>(tiff ? ctx->stream_chunk_tiff : ctx->stream_chunk, n_targets);
    // the two-kernel TIFF path addresses the chunk's decoded pixels with 32 bits
    if (tiff && !fused_ingest) chunk = std::min<int64_t>(chunk, std::max<int64_t>(1, (int64_t) (0xF0000000ull / img_bytes)));
    // the chunk plan: (device, first target, count); host targets go round-robin over the devices, a resident library is
    // walked shard by shard (first = index LOCAL to the shard)
    struct Chunk { int d; int64_t first, cnt; };
    std::vector<Chunk> plan;
    if (resident) {
        int64_t longest = 0;
        for (int d = 0; d < D; d++) longest = std::max(longest, resident->local_size(d));
        for (int64_t f = 0; f < longest; f += chunk)
            for (int d = 0; d < D; d++)
                if (f < resident->local_size(d)) plan.push_back({d, f, std::min<int64_t>(chunk, resident->local_size(d) - f)});
    } else {
        for (const StreamChunk &pc : stream_chunk_plan(D, n_targets, chunk, tiff ? tiff->offsets : nullptr, (uint64_t) ctx->stream_chunk_bytes))
            plan.push_back({pc.d, pc.first, pc.cnt});
    }
    const int64_t n_chunks = (int64_t) plan.size();
    const int thr = ms->params.data_threshold;
    const int rings = ms->params.xy_shift / 2;
    const bool want_occ = batched_kernel_supported(ms->params.xy_shift, g) && M >= band_min_masks();

    size_t tiff_comp_bytes = 0;
    std::vector<TiffStrip> strips;
    if (tiff) {
        for (const Chunk &ch : plan) {
            const int64_t a = tiff->offsets[ch.first], b = tiff->offsets[ch.first + ch.cnt];
            if (a < 0 || b < a) return ctx->fail(CDS_ERR_BAD_ARG, "cds_search_stream_tiff: offsets must be non-decreasing");
            tiff_comp_bytes = std::max(tiff_comp_bytes, (size_t) (b - a) + 64);
        }
    }

    std::vector<int32_t> min_score(M);
    for (int m = 0; m < M; m++) min_score[m] = min_matching_score(ms->sizes[m], pct_positive_pixels);
    const int used_devs = resident ? D : (int) std::min<int64_t>(D, n_chunks);
    // entries of a device's list of passing pairs
    const int64_t list_cap = best ? ctx->best_list_bytes / kBestPairBytes : all ? all->capacity : 0;
    std::vector<uint64_t *> all_keys(D, nullptr);
    std::vector<int32_t *> all_masks(D, nullptr);
    std::vector<unsigned long long *> all_counter(D, nullptr);
    std::vector<DevGroups> groups(D);          // best: the targets' group keys on every device
    std::vector<void *> gathered;              // best, several devices: the lists moved to the first device
    auto release_all = [&]() {
        for (int d = 0; d < D; d++) {
            if (!all_keys[d] && !all_masks[d] && !all_counter[d] && !groups[d].line && !(d == 0 && !gathered.empty())) continue;
            cudaSetDevice(ctx->devs[d].dev);
            cudaStreamSynchronize(ctx->devs[d].stream);
            ctx->devs[d].pool.free(all_keys[d]);
            ctx->devs[d].pool.free(all_masks[d]);
            ctx->devs[d].pool.free(all_counter[d]);
            groups[d].release(ctx->devs[d]);
            if (d == 0) for (void *p : gathered) ctx->devs[0].pool.free(p);
        }
    };
    struct Releaser { std::function<void()> f; ~Releaser() { f(); } } releaser{release_all};
    for (int d = 0; d < used_devs; d++) {
        DevState &ds = ctx->devs[d];
        CDS_TRY(ensure_stream_bufs(ctx, ds, g, bpitch, chunk, M, k, resident == nullptr, resident ? 0 : (tiff ? (fused_ingest ? 0 : 1) : 2)));
        if (tiff) CDS_TRY(ensure_tiff_bufs(ctx, ds, tiff_comp_bytes, (size_t) chunk * 128));
        CDS_CUDA(ctx, cudaMemcpyAsync(ds.sb.min_score, min_score.data(), (size_t) M * sizeof(int32_t), cudaMemcpyHostToDevice, ds.stream));
        CDS_CUDA(ctx, cudaMemsetAsync(ds.sb.counts_run, 0, (size_t) M * sizeof(int32_t), ds.stream));
        if (best) CDS_TRY(upload_target_groups(ctx, ds, best->groups, n_targets, groups[d]));
        if (collect) {
            const size_t cap = (size_t) std::max<int64_t>(list_cap, 1);
            CDS_CUDA(ctx, ds.pool.alloc((void **) &all_keys[d], cap * sizeof(uint64_t)));
            CDS_CUDA(ctx, ds.pool.alloc((void **) &all_masks[d], cap * sizeof(int32_t)));
            CDS_CUDA(ctx, ds.pool.alloc((void **) &all_counter[d], sizeof(unsigned long long)));
            CDS_CUDA(ctx, cudaMemsetAsync(all_counter[d], 0, sizeof(unsigned long long), ds.stream));
        }
        CDS_CUDA(ctx, cudaEventRecord(ds.ev0, ds.stream));
        const size_t need = (size_t) 2 * (n_chunks / std::max(used_devs, 1) + 2);
        while (ds.sb.timing.size() < need) {
            cudaEvent_t e;
            CDS_CUDA(ctx, cudaEventCreate(&e));
            ds.sb.timing.push_back(e);
        }
    }

    // whatever way this call ends (a bad file in chunk 5, a CUDA error), nothing of it is still in flight afterwards: the next
    // call reuses the staging buffers from chunk 0 without waiting for anybody
    struct Drain {
        cds_ctx *ctx; int n;
        ~Drain() {
            for (int d = 0; d < n; d++) {
                cudaSetDevice(ctx->devs[d].dev);
                if (ctx->devs[d].sb.copy_stream) cudaStreamSynchronize(ctx->devs[d].sb.copy_stream);
                cudaStreamSynchronize(ctx->devs[d].stream);
            }
        }
    } drain{ctx, used_devs};

    // profiling aid (CDSGPU_STREAM_TRACE=1): device events around every phase of every chunk and the host's own clock, printed to
    // stderr when the call ends
    static const bool trace = std::getenv("CDSGPU_STREAM_TRACE") != nullptr;
    struct ChunkTrace { int d; int64_t cnt; cudaEvent_t ev[5]; double host_parse_ms, host_wait_ms, host_enqueue_at_ms; };
    std::vector<ChunkTrace> traces;
    const auto t_host0 = std::chrono::steady_clock::now();
    auto host_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_host0).count(); };
    auto mark = [&](ChunkTrace *tr, int i, cudaStream_t st) {
        if (!tr) return;
        cudaEventCreate(&tr->ev[i]);
        cudaEventRecord(tr->ev[i], st);
    };

    // best, with a per-sample limit: a device's list is compacted exactly (bestsel_compact) when the next chunk might not fit.  bound[d]
    // = most pairs the list can hold by now (a chunk adds at most masks x targets); only when it passes the budget does the host wait
    // for the true count.  Without a limit the list cannot shrink and a list that overflows fails at the end, with the size it needs.
    std::vector<int64_t> bound(D, 0), compacted_at(D, -1);
    auto read_count = [&](int d, int64_t &n) -> cds_status {
        unsigned long long c = 0;
        CDS_CUDA(ctx, cudaMemcpyAsync(&c, all_counter[d], sizeof c, cudaMemcpyDeviceToHost, ctx->devs[d].stream));
        CDS_CUDA(ctx, cudaStreamSynchronize(ctx->devs[d].stream));
        ctx->stats.d2h_bytes += (int64_t) sizeof c;
        n = (int64_t) c;
        return CDS_OK;
    };
    auto best_make_room = [&](int d, int64_t most) -> cds_status {
        if (bound[d] + most <= list_cap) return CDS_OK;
        int64_t n = 0;
        CDS_TRY(read_count(d, n));
        if (n + most > list_cap && n != compacted_at[d]) {
            // a resident library's keys are still shard-local here
            CDS_TRY(bestsel_compact(ctx, ctx->devs[d], all_keys[d], all_masks[d], n, all_counter[d], groups[d], best->top_matches_per_sample,
                                    resident ? d : 0, resident ? D : 1));
            compacted_at[d] = n;
            CDS_CUDA(ctx, cudaSetDevice(ctx->devs[d].dev));
        }
        bound[d] = n;
        return CDS_OK;
    };
    auto best_check = [&](int d, int64_t most) -> cds_status {
        bound[d] += most;
        if (bound[d] <= list_cap) return CDS_OK;
        int64_t n = 0;
        CDS_TRY(read_count(d, n));
        if (n > list_cap) {
            char buf[300];
            snprintf(buf, sizeof buf, "best matches: the passing pairs of device %d need at least %lld bytes after keeping %d per sample; "
                     "\"best_list_bytes\" is %lld", d, (long long) (n * kBestPairBytes), best->top_matches_per_sample, (long long) ctx->best_list_bytes);
            return ctx->fail(CDS_ERR_CAPACITY, buf);
        }
        bound[d] = n;
        return CDS_OK;
    };

    // enqueue every chunk; nothing below blocks the host when the source is pinned memory
    std::vector<int64_t> per_dev(D, 0);
    if (trace) traces.reserve(plan.size());
    for (const Chunk &ch : plan) {
        const int d = ch.d;
        DevState &ds = ctx->devs[d];
        StreamBufs &sb = ds.sb;
        const int64_t j = per_dev[d]++;
        const int slot = (int) (j & 1);
        const int64_t first = ch.first, cnt = ch.cnt;
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        const uint32_t *planes = sb.planes;
        cudaStream_t ist = ds.stream;             // where this chunk's ingest and occupancy kernels run
        ChunkTrace *tr = nullptr;
        if (trace) { traces.push_back(ChunkTrace{d, cnt, {}, 0, 0, 0}); tr = &traces.back(); }
        const double t_chunk0 = trace ? host_ms() : 0;
        if (resident) {
            planes = resident->shards[d].planes + (size_t) first * g.plane_stride();      // the same geometry, starting at plane `first`
        } else if (tiff) {
            // host: the chunk's strip table from the files' tags (overlaps the device's work on earlier chunks)
            strips.clear();
            const int64_t base = tiff->offsets[first];
            std::string err;
            for (int64_t i = 0; i < cnt; i++) {
                const int64_t a = tiff->offsets[first + i], b = tiff->offsets[first + i + 1];
                if (b < a) return ctx->fail(CDS_ERR_BAD_ARG, "cds_search_stream_tiff: offsets must be non-decreasing");
                cds_status st = tiff_collect_strips(tiff->blob + a, (size_t) (b - a), g.W, g.H, (uint64_t) (a - base),
                                                    fused_ingest ? (uint64_t) i * g.H : (uint64_t) i * img_bytes, strips, err, fused_ingest);
                if (st != CDS_OK) return ctx->fail(st, "cds_search_stream_tiff: file " + std::to_string(first + i) + ": " + err);
            }
            CDS_TRY(ensure_tiff_bufs(ctx, ds, tiff_comp_bytes, strips.size()));
            const double t_parsed = trace ? host_ms() : 0;
            if (j >= 2) CDS_CUDA(ctx, cudaEventSynchronize(sb.h2d_done[slot]));        // the slot's previous table has left the host
            if (tr) { tr->host_parse_ms = t_parsed - t_chunk0; tr->host_wait_ms = host_ms() - t_parsed; }
            memcpy(sb.h_strips[slot], strips.data(), strips.size() * sizeof(TiffStrip));
            if (j >= 2) CDS_CUDA(ctx, cudaStreamWaitEvent(sb.copy_stream, sb.enc_done[slot], 0));
            const size_t bytes = (size_t) (tiff->offsets[first + cnt] - base);
            CDS_CUDA(ctx, cudaMemcpyAsync(sb.comp[slot], tiff->blob + base, bytes, cudaMemcpyHostToDevice, sb.copy_stream));
            CDS_CUDA(ctx, cudaMemcpyAsync(sb.d_strips[slot], sb.h_strips[slot], strips.size() * sizeof(TiffStrip), cudaMemcpyHostToDevice, sb.copy_stream));
            ctx->stats.h2d_bytes += (int64_t) bytes + (int64_t) (strips.size() * sizeof(TiffStrip));
            CDS_CUDA(ctx, cudaEventRecord(sb.h2d_done[slot], sb.copy_stream));
            mark(tr, 0, ds.stream);                  // the compute stream's position BEFORE it waits for the upload
            if (descs_pending) ist = sb.copy_stream;          // (this chunk's preprocessing runs beside the list build, see above)
            if (ist == ds.stream) CDS_CUDA(ctx, cudaStreamWaitEvent(ds.stream, sb.h2d_done[slot], 0));
            mark(tr, 1, ds.stream);
            if (fused_ingest) {
                // strips -> code words + per-sector valid bits in one kernel, no RGB image in HBM in between
                launch_tiff_encode(sb.comp[slot], (const TiffStrip *) sb.d_strips[slot], (int64_t) strips.size(), sb.planes, g, 0, ds.d_rank_tab, thr,
                                   want_occ ? sb.valid : nullptr, sb.strip_counter, ist);
                ctx->stats.kernel_launches += 1;
            } else {
                // decode into one RGB area (stream order protects it), then the usual encoder
                launch_tiff_decode(sb.comp[slot], (const TiffStrip *) sb.d_strips[slot], (int64_t) strips.size(), sb.staging[0], ist);
                launch_encode_rgb(sb.staging[0], cnt, sb.planes, g, 0, ds.d_rank_tab, thr, ist, want_occ ? sb.valid : nullptr);
                ctx->stats.kernel_launches += 2;
            }
            CDS_CUDA(ctx, cudaEventRecord(sb.enc_done[slot], ist));
            mark(tr, 2, ds.stream);
        } else {
            if (j >= 2) CDS_CUDA(ctx, cudaStreamWaitEvent(sb.copy_stream, sb.enc_done[slot], 0));
            CDS_CUDA(ctx, cudaMemcpyAsync(sb.staging[slot], targets_rgb + (size_t) first * img_bytes, (size_t) cnt * img_bytes,
                                         cudaMemcpyHostToDevice, sb.copy_stream));
            ctx->stats.h2d_bytes += (int64_t) cnt * (int64_t) img_bytes;
            CDS_CUDA(ctx, cudaEventRecord(sb.h2d_done[slot], sb.copy_stream));
            CDS_CUDA(ctx, cudaStreamWaitEvent(ds.stream, sb.h2d_done[slot], 0));
            launch_encode_rgb(sb.staging[slot], cnt, sb.planes, g, 0, ds.d_rank_tab, thr, ds.stream, want_occ ? sb.valid : nullptr);
            CDS_CUDA(ctx, cudaEventRecord(sb.enc_done[slot], ds.stream));
            ctx->stats.kernel_launches++;
        }
        TargetView tv;
        tv.planes = planes; tv.g = g; tv.bpitch = bpitch; tv.n = cnt; tv.occ = nullptr; tv.occ_ready = false;
        if (want_occ) {
            // host targets: the encoder has just written the valid bits of this chunk
            launch_occupancy(planes, g, 0, cnt, rings, bpitch, sb.valid, sb.chunk, sb.occ, ist, resident == nullptr);
            ctx->stats.kernel_launches += resident ? 2 : 1;      // (valid bits,) occupancy incl. the non-empty bits
            tv.occ = sb.occ;
            tv.occ_ready = true;
        }
        CDS_CUDA(ctx, cudaGetLastError());
        if (ist != ds.stream) {
            // the lists, now; then the compute stream joins the side stream
            cudaEvent_t pre = sb.h2d_done[slot ^ 1];          // (free: no chunk of this device has used the other slot yet)
            CDS_CUDA(ctx, cudaEventRecord(pre, ist));
            CDS_TRY(ms->sync_descs());
            descs_pending = false;
            CDS_CUDA(ctx, cudaSetDevice(ds.dev));
            CDS_CUDA(ctx, cudaStreamWaitEvent(ds.stream, pre, 0));
        }
        if (tr && tiff) mark(tr, 3, ds.stream);
        CDS_TRY(launch_match_view(ctx, ms, tv, d, 0, M, sb.scores, ds.stream, sb.timing[2 * j], sb.timing[2 * j + 1]));
        if (collect) {
            const bool compacting = best && best->top_matches_per_sample > 0;
            if (compacting) CDS_TRY(best_make_room(d, (int64_t) M * cnt));
            launch_collect_matches(sb.scores, M, cnt, sb.min_score, 0, first, all_keys[d], all_masks[d], all_counter[d],
                                   (unsigned long long) list_cap, ds.stream);
            ctx->stats.kernel_launches++;
            if (compacting) CDS_TRY(best_check(d, (int64_t) M * cnt));
        } else {
            launch_topk(sb.scores, M, cnt, sb.min_score, k, first, sb.keys_chunk, sb.counts_chunk, ds.stream);
            launch_topk_merge(sb.keys_run, sb.counts_run, sb.keys_chunk, sb.counts_chunk, M, k, ds.stream);
            ctx->stats.kernel_launches += 2;
        }
        if (tr && tiff) { mark(tr, 4, ds.stream); tr->host_enqueue_at_ms = host_ms(); }
        CDS_CUDA(ctx, cudaGetLastError());
    }

    // read the per-device lists back and merge them (no collective: nothing is reduced across devices)
    const size_t keys_bytes = (size_t) M * k * sizeof(uint64_t);
    std::vector<unsigned long long> all_n(D, 0);
    for (int d = 0; d < used_devs; d++) {
        DevState &ds = ctx->devs[d];
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        CDS_CUDA(ctx, cudaEventRecord(ds.ev2, ds.stream));
        if (collect) {
            CDS_CUDA(ctx, cudaMemcpyAsync(&all_n[d], all_counter[d], sizeof(unsigned long long), cudaMemcpyDeviceToHost, ds.stream));
            continue;
        }
        CDS_TRY(ctx->ensure_pinned(ds, keys_bytes + (size_t) M * sizeof(int32_t)));
        uint8_t *hp = (uint8_t *) ds.h_pinned;
        CDS_CUDA(ctx, cudaMemcpyAsync(hp, ds.sb.keys_run, keys_bytes, cudaMemcpyDeviceToHost, ds.stream));
        CDS_CUDA(ctx, cudaMemcpyAsync(hp + keys_bytes, ds.sb.counts_run, (size_t) M * sizeof(int32_t), cudaMemcpyDeviceToHost, ds.stream));
        ctx->stats.d2h_bytes += (int64_t) keys_bytes + (int64_t) M * 4;
    }
    double match_ms = 0, total_ms = 0;
    for (int d = 0; d < used_devs; d++) {
        DevState &ds = ctx->devs[d];
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
        float ms_f = 0;
        double dev_match = 0;
        for (int64_t j = 0; j < per_dev[d]; j++) {
            cudaEventElapsedTime(&ms_f, ds.sb.timing[2 * j], ds.sb.timing[2 * j + 1]);
            dev_match += ms_f;
        }
        match_ms = std::max(match_ms, dev_match);
        cudaEventElapsedTime(&ms_f, ds.ev0, ds.ev2);
        total_ms = std::max(total_ms, (double) ms_f);
    }
    if (trace && tiff) {
        std::fprintf(stderr, "# chunk dev targets | host: parse wait enqueued_at | device: start(since ev0) wait_h2d ingest occupancy match topk | match events\n");
        std::vector<int64_t> jj(D, 0);
        for (size_t c = 0; c < traces.size(); c++) {
            ChunkTrace &t = traces[c];
            float a0 = 0, w = 0, ing = 0, occm = 0, rest = 0, mm = 0;
            cudaEventElapsedTime(&a0, ctx->devs[t.d].ev0, t.ev[0]);
            cudaEventElapsedTime(&w, t.ev[0], t.ev[1]);
            cudaEventElapsedTime(&ing, t.ev[1], t.ev[2]);
            cudaEventElapsedTime(&occm, t.ev[2], t.ev[3]);
            cudaEventElapsedTime(&rest, t.ev[3], t.ev[4]);
            const int64_t j = jj[t.d]++;
            cudaEventElapsedTime(&mm, ctx->devs[t.d].sb.timing[2 * j], ctx->devs[t.d].sb.timing[2 * j + 1]);
            std::fprintf(stderr, "%3zu %d %5lld | %7.3f %7.3f %8.3f | %8.3f %7.3f %7.3f %7.3f %7.3f %7.3f\n", c, t.d, (long long) t.cnt, t.host_parse_ms, t.host_wait_ms,
                         t.host_enqueue_at_ms, a0, w, ing, occm, mm, rest - mm);
            for (int i = 0; i < 5; i++) cudaEventDestroy(t.ev[i]);
        }
    }
    ctx->stats.match_kernel_ms = match_ms;
    ctx->stats.total_device_ms = total_ms;
    ctx->stats.comparisons = (int64_t) M * n_targets;
    ctx->stats.chunked = 1;
    if (best) {
        // the selection runs where all of a mask's pairs are: the first device; only the selected pairs and their count come back
        std::vector<int64_t> n_dev(used_devs);
        for (int d = 0; d < used_devs; d++) {
            ctx->stats.d2h_bytes += (int64_t) sizeof(unsigned long long);
            n_dev[d] = (int64_t) all_n[d];
            if (n_dev[d] > list_cap) {
                char buf[300];
                snprintf(buf, sizeof buf, "best matches: %lld pairs pass isMatch on device %d, their list needs %lld bytes; \"best_list_bytes\" is %lld%s",
                         (long long) n_dev[d], d, (long long) (n_dev[d] * kBestPairBytes), (long long) ctx->best_list_bytes,
                         best->top_matches_per_sample > 0 ? "" : " (without a per-sample limit the list cannot be compacted)");
                return ctx->fail(CDS_ERR_CAPACITY, buf);
            }
        }
        for (int d = 0; d < used_devs; d++) {
            DevState &ds = ctx->devs[d];
            CDS_CUDA(ctx, cudaSetDevice(ds.dev));
            if (resident) launch_bestsel_globalize(all_keys[d], n_dev[d], d, D, ds.stream);
            CDS_CUDA(ctx, cudaGetLastError());
            if (used_devs > 1)
                CDS_TRY(bestsel_compact(ctx, ds, all_keys[d], all_masks[d], n_dev[d], all_counter[d], groups[d], best->top_matches_per_sample, 0, 1));
        }
        DevState &d0 = ctx->devs[0];
        uint64_t *keys = all_keys[0];
        int32_t *masks = all_masks[0];
        int64_t n = n_dev[0];
        if (used_devs > 1) {
            for (int d = 1; d < used_devs; d++) n += n_dev[d];
            for (int d = 0; d < used_devs; d++) {
                CDS_CUDA(ctx, cudaSetDevice(ctx->devs[d].dev));
                CDS_CUDA(ctx, cudaStreamSynchronize(ctx->devs[d].stream));
            }
            CDS_CUDA(ctx, cudaSetDevice(d0.dev));
            void *gk = nullptr, *gm = nullptr;
            CDS_CUDA(ctx, d0.pool.alloc(&gk, (size_t) std::max<int64_t>(n, 1) * sizeof(uint64_t)));
            gathered.push_back(gk);
            CDS_CUDA(ctx, d0.pool.alloc(&gm, (size_t) std::max<int64_t>(n, 1) * sizeof(int32_t)));
            gathered.push_back(gm);
            keys = (uint64_t *) gk;
            masks = (int32_t *) gm;
            int64_t at = 0;
            for (int d = 0; d < used_devs; d++) {
                DevState &src = ctx->devs[d];
                const struct { void *dst; const void *src; size_t bytes; } parts[] = {
                    {keys + at, all_keys[d], (size_t) n_dev[d] * sizeof(uint64_t)}, {masks + at, all_masks[d], (size_t) n_dev[d] * sizeof(int32_t)}};
                at += n_dev[d];
                int peer = 0;
                if (src.dev != d0.dev) CDS_CUDA(ctx, cudaDeviceCanAccessPeer(&peer, d0.dev, src.dev));
                for (const auto &pt : parts) {
                    if (pt.bytes == 0) continue;
                    if (src.dev == d0.dev) {
                        CDS_CUDA(ctx, cudaMemcpyAsync(pt.dst, pt.src, pt.bytes, cudaMemcpyDeviceToDevice, d0.stream));
                    } else if (peer) {
                        CDS_CUDA(ctx, cudaMemcpyPeerAsync(pt.dst, d0.dev, pt.src, src.dev, pt.bytes, d0.stream));
                    } else {
                        // no peer access: staged through pinned host memory
                        CDS_TRY(ctx->ensure_pinned(src, pt.bytes));
                        CDS_CUDA(ctx, cudaSetDevice(src.dev));
                        CDS_CUDA(ctx, cudaMemcpyAsync(src.h_pinned, pt.src, pt.bytes, cudaMemcpyDeviceToHost, src.stream));
                        CDS_CUDA(ctx, cudaStreamSynchronize(src.stream));
                        CDS_CUDA(ctx, cudaSetDevice(d0.dev));
                        CDS_CUDA(ctx, cudaMemcpyAsync(pt.dst, src.h_pinned, pt.bytes, cudaMemcpyHostToDevice, d0.stream));
                        CDS_CUDA(ctx, cudaStreamSynchronize(d0.stream));
                        ctx->stats.d2h_bytes += (int64_t) pt.bytes;
                        ctx->stats.h2d_bytes += (int64_t) pt.bytes;
                    }
                }
            }
        }
        BestSelOut o;
        o.capacity = best->capacity;
        o.mask = best->mask; o.target = best->target; o.score = best->score; o.mirrored = best->mirrored;
        o.count = best->count;
        return bestsel_select(ctx, d0, keys, masks, n, M, false, groups[0], best->top_lines, best->top_samples_per_line,
                              best->top_matches_per_sample, o);
    }
    if (all) {
        // every passing pair, ordered like the reference's writer: by mask, descending matchingPixels, ascending target
        uint64_t total = 0;
        for (int d = 0; d < used_devs; d++) total += all_n[d];
        *all->count = (int64_t) total;
        if (total > (uint64_t) all->capacity) {
            char buf[160];
            snprintf(buf, sizeof buf, "cds_search_stream_matches_rgb: %llu pairs pass isMatch, capacity is %lld", (unsigned long long) total, (long long) all->capacity);
            return ctx->fail(CDS_ERR_CAPACITY, buf);
        }
        struct Pair { int32_t mask; uint64_t key; };
        std::vector<Pair> pairs;
        pairs.reserve(total);
        std::vector<uint64_t> hk;
        std::vector<int32_t> hm;
        for (int d = 0; d < used_devs; d++) {
            const size_t n = (size_t) all_n[d];
            if (!n) continue;
            hk.resize(n); hm.resize(n);
            CDS_CUDA(ctx, cudaSetDevice(ctx->devs[d].dev));
            CDS_CUDA(ctx, cudaMemcpy(hk.data(), all_keys[d], n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
            CDS_CUDA(ctx, cudaMemcpy(hm.data(), all_masks[d], n * sizeof(int32_t), cudaMemcpyDeviceToHost));
            ctx->stats.d2h_bytes += (int64_t) (n * 12);
            for (size_t i = 0; i < n; i++) {
                uint64_t key = hk[i];
                if (resident) {       // keys of a resident library carry shard-local indices
                    int32_t sc; int64_t tg; uint8_t mir;
                    topk_decode_key(key, sc, tg, mir);
                    key = topk_make_key(sc, resident->global_of(d, tg), mir);
                }
                pairs.push_back({hm[i], key});
            }
        }
        std::sort(pairs.begin(), pairs.end(), [](const Pair &a, const Pair &b) { return a.mask != b.mask ? a.mask < b.mask : a.key < b.key; });
        for (size_t i = 0; i < pairs.size(); i++) {
            int32_t sc; int64_t tg; uint8_t mir;
            topk_decode_key(pairs[i].key, sc, tg, mir);
            all->mask[i] = pairs[i].mask;
            all->target[i] = tg;
            all->score[i] = sc;
            if (all->mirrored) all->mirrored[i] = mir;
        }
        return CDS_OK;
    }
    struct Item { int32_t score; int64_t target; uint8_t mir; };
    std::vector<Item> items;
    for (int m = 0; m < M; m++) {
        items.clear();
        for (int d = 0; d < used_devs; d++) {
            const uint8_t *hp = (const uint8_t *) ctx->devs[d].h_pinned;
            const uint64_t *keys = (const uint64_t *) hp + (size_t) m * k;
            const int c = std::min(((const int32_t *) (hp + keys_bytes))[m], k);
            for (int i = 0; i < c; i++) {
                Item it;
                topk_decode_key(keys[i], it.score, it.target, it.mir);
                if (resident) it.target = resident->global_of(d, it.target);
                items.push_back(it);
            }
        }
        if (used_devs > 1)
            std::sort(items.begin(), items.end(), [](const Item &a, const Item &b) {
                if (a.score != b.score) return a.score > b.score;
                return a.target < b.target;
            });
        const int c = (int) std::min<size_t>(items.size(), (size_t) k);
        out_count[m] = c;
        for (int i = 0; i < c; i++) {
            out_score[(size_t) m * k + i] = items[i].score;
            out_target[(size_t) m * k + i] = items[i].target;
            if (out_mirrored) out_mirrored[(size_t) m * k + i] = items[i].mir;
        }
    }
    return CDS_OK;
}

}  // namespace

extern "C" cds_status cds_search_stream_rgb(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *targets_rgb, int64_t n_targets,
                                            int32_t k, double pct_positive_pixels,
                                            int32_t *out_score, int64_t *out_target, uint8_t *out_mirrored, int32_t *out_count)
{
    return cds::abi_guard("cds_search_stream_rgb", [&]() -> cds_status {
        if (!ctx || !ms) { set_tls_error("cds_search_stream_rgb: NULL argument"); return CDS_ERR_BAD_ARG; }
        return stream_search_impl(ctx, ms, targets_rgb, n_targets, k, pct_positive_pixels, out_score, out_target, out_mirrored, out_count, nullptr, nullptr);
    });
}

extern "C" cds_status cds_search_stream_matches_rgb(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *targets_rgb, int64_t n_targets,
                                                    double pct_positive_pixels, int64_t capacity,
                                                    int32_t *out_mask, int64_t *out_target, int32_t *out_score, uint8_t *out_mirrored,
                                                    int64_t *out_count)
{
    return cds::abi_guard("cds_search_stream_matches_rgb", [&]() -> cds_status {
        if (!ctx || !ms) { set_tls_error("cds_search_stream_matches_rgb: NULL argument"); return CDS_ERR_BAD_ARG; }
        const AllMatchesOut all{capacity, out_mask, out_target, out_score, out_mirrored, out_count};
        return stream_search_impl(ctx, ms, targets_rgb, n_targets, 1, pct_positive_pixels, nullptr, nullptr, nullptr, nullptr, &all, nullptr);
    });
}

extern "C" cds_status cds_search_stream_tiff(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *blob, const int64_t *offsets, int64_t n_targets,
                                             int32_t k, double pct_positive_pixels,
                                             int32_t *out_score, int64_t *out_target, uint8_t *out_mirrored, int32_t *out_count)
{
    return cds::abi_guard("cds_search_stream_tiff", [&]() -> cds_status {
        if (!ctx || !ms) { set_tls_error("cds_search_stream_tiff: NULL argument"); return CDS_ERR_BAD_ARG; }
        const TiffSource src{blob, offsets};
        return stream_search_impl(ctx, ms, nullptr, n_targets, k, pct_positive_pixels, out_score, out_target, out_mirrored, out_count, nullptr, nullptr, &src);
    });
}

extern "C" cds_status cds_search_stream_matches_tiff(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *blob, const int64_t *offsets, int64_t n_targets,
                                                     double pct_positive_pixels, int64_t capacity,
                                                     int32_t *out_mask, int64_t *out_target, int32_t *out_score, uint8_t *out_mirrored,
                                                     int64_t *out_count)
{
    return cds::abi_guard("cds_search_stream_matches_tiff", [&]() -> cds_status {
        if (!ctx || !ms) { set_tls_error("cds_search_stream_matches_tiff: NULL argument"); return CDS_ERR_BAD_ARG; }
        const AllMatchesOut all{capacity, out_mask, out_target, out_score, out_mirrored, out_count};
        const TiffSource src{blob, offsets};
        return stream_search_impl(ctx, ms, nullptr, n_targets, 1, pct_positive_pixels, nullptr, nullptr, nullptr, nullptr, &all, nullptr, &src);
    });
}

// The same chunked search over a device-resident library: occupancy bitmaps are built per chunk instead of being kept for
// the whole library (cds_search_topk uses this when they do not fit next to the code planes, e.g. 50 000 targets per GPU).
namespace cds {
cds_status search_library_chunked(cds_ctx *ctx, const cds_maskset *ms, cds_library *lib, int32_t k, double pct_positive_pixels,
                                  int32_t *out_score, int64_t *out_target, uint8_t *out_mirrored, int32_t *out_count)
{
    return stream_search_impl(ctx, ms, nullptr, 0, k, pct_positive_pixels, out_score, out_target, out_mirrored, out_count, nullptr, lib);
}
}  // namespace cds

extern "C" cds_status cds_search_matches(cds_ctx *ctx, const cds_maskset *ms, cds_library *lib, double pct_positive_pixels, int64_t capacity,
                                         int32_t *out_mask, int64_t *out_target, int32_t *out_score, uint8_t *out_mirrored, int64_t *out_count)
{
    return cds::abi_guard("cds_search_matches", [&]() -> cds_status {
        if (!ctx || !ms || !lib) { set_tls_error("cds_search_matches: NULL argument"); return CDS_ERR_BAD_ARG; }
        if (ms->W != lib->g.W || ms->H != lib->g.H) {
            std::lock_guard<std::recursive_mutex> lk(ctx->mu);
            char buf[200];
            snprintf(buf, sizeof buf, "Invalid image size - target's image size (%d, %d) must match query's image size: (%d, %d)", ms->W, ms->H, lib->g.W, lib->g.H);
            return ctx->fail(CDS_ERR_SIZE_MISMATCH, buf);
        }
        const AllMatchesOut all{capacity, out_mask, out_target, out_score, out_mirrored, out_count};
        return stream_search_impl(ctx, ms, nullptr, 0, 1, pct_positive_pixels, nullptr, nullptr, nullptr, nullptr, &all, lib);
    });
}

// The best-matches searches: the same collection of passing pairs, then ColorMIPProcessUtils.selectBestMatches per mask on the
// device (csrc/cds_bestsel.cu).  The groups are checked before anything touches a device.
namespace {
cds_status best_matches_entry(const char *name, cds_ctx *ctx, const cds_maskset *ms, int64_t n_targets, const cds_target_groups *groups,
                              const std::function<cds_status()> &run)
{
    const std::string err = cds::check_target_groups(groups, std::max<int64_t>(n_targets, 0));
    if (!err.empty()) {
        if (!ctx) { set_tls_error(std::string(name) + ": " + err); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        return ctx->fail(CDS_ERR_BAD_ARG, std::string(name) + ": " + err);
    }
    if (!ctx || !ms) { set_tls_error(std::string(name) + ": NULL argument"); return CDS_ERR_BAD_ARG; }
    return run();
}
}  // namespace

extern "C" cds_status cds_search_best_matches(cds_ctx *ctx, const cds_maskset *ms, cds_library *lib, const cds_target_groups *groups,
                                              double pct_positive_pixels, int32_t top_lines, int32_t top_samples_per_line, int32_t top_matches_per_sample,
                                              int64_t capacity, int32_t *out_mask, int64_t *out_target, int32_t *out_score, uint8_t *out_mirrored,
                                              int64_t *out_count)
{
    return cds::abi_guard("cds_search_best_matches", [&]() -> cds_status {
        if (!lib) { set_tls_error("cds_search_best_matches: NULL argument"); return CDS_ERR_BAD_ARG; }
        return best_matches_entry("cds_search_best_matches", ctx, ms, lib->size, groups, [&]() -> cds_status {
            if (ms->W != lib->g.W || ms->H != lib->g.H) {
                std::lock_guard<std::recursive_mutex> lk(ctx->mu);
                char buf[200];
                snprintf(buf, sizeof buf, "Invalid image size - target's image size (%d, %d) must match query's image size: (%d, %d)", ms->W, ms->H, lib->g.W, lib->g.H);
                return ctx->fail(CDS_ERR_SIZE_MISMATCH, buf);
            }
            const BestMatchesOut best{groups, top_lines, top_samples_per_line, top_matches_per_sample, capacity, out_mask, out_target, out_score, out_mirrored, out_count};
            return stream_search_impl(ctx, ms, nullptr, 0, 1, pct_positive_pixels, nullptr, nullptr, nullptr, nullptr, nullptr, lib, nullptr, &best);
        });
    });
}

extern "C" cds_status cds_search_stream_best_matches_tiff(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *blob, const int64_t *offsets,
                                                          int64_t n_targets, const cds_target_groups *groups, double pct_positive_pixels,
                                                          int32_t top_lines, int32_t top_samples_per_line, int32_t top_matches_per_sample,
                                                          int64_t capacity, int32_t *out_mask, int64_t *out_target, int32_t *out_score,
                                                          uint8_t *out_mirrored, int64_t *out_count)
{
    return cds::abi_guard("cds_search_stream_best_matches_tiff", [&]() -> cds_status {
        return best_matches_entry("cds_search_stream_best_matches_tiff", ctx, ms, n_targets, groups, [&]() -> cds_status {
            const BestMatchesOut best{groups, top_lines, top_samples_per_line, top_matches_per_sample, capacity, out_mask, out_target, out_score, out_mirrored, out_count};
            const TiffSource src{blob, offsets};
            return stream_search_impl(ctx, ms, nullptr, n_targets, 1, pct_positive_pixels, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, &src, &best);
        });
    });
}

extern "C" cds_status cds_search_stream_best_matches_rgb(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *targets_rgb, int64_t n_targets,
                                                         const cds_target_groups *groups, double pct_positive_pixels,
                                                         int32_t top_lines, int32_t top_samples_per_line, int32_t top_matches_per_sample,
                                                         int64_t capacity, int32_t *out_mask, int64_t *out_target, int32_t *out_score,
                                                         uint8_t *out_mirrored, int64_t *out_count)
{
    return cds::abi_guard("cds_search_stream_best_matches_rgb", [&]() -> cds_status {
        return best_matches_entry("cds_search_stream_best_matches_rgb", ctx, ms, n_targets, groups, [&]() -> cds_status {
            const BestMatchesOut best{groups, top_lines, top_samples_per_line, top_matches_per_sample, capacity, out_mask, out_target, out_score, out_mirrored, out_count};
            return stream_search_impl(ctx, ms, targets_rgb, n_targets, 1, pct_positive_pixels, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, &best);
        });
    });
}

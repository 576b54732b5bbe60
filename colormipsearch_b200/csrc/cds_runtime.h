// cds_runtime.h -- host-side object model behind the C ABI (include/cdsgpu.h).  Internal.
#ifndef CDS_RUNTIME_H
#define CDS_RUNTIME_H

#include <cstdlib>
#include <cuda_runtime.h>

#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/cdsgpu.h"
#include "cds_common.h"
#include "cds_kernels.cuh"
#include "cds_tables.h"

namespace cds {

constexpr int64_t kLibBlock = 64;   // targets per block of the block-cyclic device sharding

// Device buffers of the streaming search (cds_search_stream_rgb), kept between calls.
struct StreamBufs {
    int W = 0, H = 0;
    int64_t chunk = 0;                  // targets per chunk the buffers are sized for
    int64_t m_cap = 0, key_cap = 0;     // masks / (masks * k) the score and key buffers are sized for
    cudaStream_t copy_stream = nullptr;
    size_t staging_cap[2] = {0, 0};
    unsigned long long *strip_counter = nullptr;   // the fused ingest kernel's work counter
    uint8_t *staging[2] = {nullptr, nullptr};   // RGB chunks as uploaded (double buffered: the next upload overlaps this chunk's kernels)
    uint32_t *planes = nullptr, *occ = nullptr, *valid = nullptr;
    int32_t *scores = nullptr;          // [masks][chunk]
    uint64_t *keys_chunk = nullptr, *keys_run = nullptr;
    int32_t *counts_chunk = nullptr, *counts_run = nullptr, *min_score = nullptr;
    cudaEvent_t h2d_done[2] = {nullptr, nullptr}, enc_done[2] = {nullptr, nullptr};
    std::vector<cudaEvent_t> timing;    // pairs around every chunk's match kernel
    // targets that arrive as TIFF files (cds_search_stream_tiff): file bytes as uploaded + strip tables, double buffered
    uint8_t *comp[2] = {nullptr, nullptr};
    void *d_strips[2] = {nullptr, nullptr}, *h_strips[2] = {nullptr, nullptr};     // cds::TiffStrip[]; the host copies are pinned
    size_t comp_cap = 0, strips_cap = 0;
    void release();
};

// Caching device allocator of one device: mask sets are created and destroyed once per batched search, and cudaMalloc /
// cudaFree cost milliseconds each (and synchronise the device).  Freed blocks are kept (up to a byte limit) and handed
// out again to requests of similar size.  Everything that uses pooled blocks runs on the device's main stream.
struct DevPool {
    std::multimap<size_t, void *> free_blocks;      // by size
    std::map<void *, size_t> live;                  // blocks handed out
    size_t cached_bytes = 0;
    cudaError_t alloc(void **p, size_t bytes);
    void free(void *p);
    void release_all();
};

struct DevState {
    int dev = -1;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;                        // uploads that overlap kernels on `stream`
    cudaEvent_t up_done[2] = {nullptr, nullptr}, up_free[2] = {nullptr, nullptr};   // double-buffered staging hand-off
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;   // match kernel start / end, search end
    uint16_t *d_rank_tab = nullptr;
    std::map<uint64_t, cds_class_interval *> d_class_tabs;   // keyed by the bits of zTolerance
    void *staging = nullptr;       // device staging for uploads
    size_t staging_bytes = 0;
    void *h_pinned = nullptr;      // pinned host scratch for read-backs
    size_t h_pinned_bytes = 0;
    void *scratch[4] = {nullptr, nullptr, nullptr, nullptr};   // grow-only device scratch (scores, min scores, keys, counts)
    size_t scratch_bytes[4] = {0, 0, 0, 0};
    StreamBufs sb;
    DevPool pool;
    MatchScratch match_scratch;       // allocated on first use (cds_ctx::ensure_match_scratch)
    uint32_t *pair_plane = nullptr;   // one code plane + one score word for cds_score_pair_rgb
    int pair_W = 0, pair_H = 0;
    uint16_t *d_slice_tab = nullptr;  // shape path: slice number of every (channel pair, max, second) (cds_shape.cu), built on first use
    std::vector<cudaEvent_t> shape_timing;   // pairs around every window's pair kernel
    void *h_pinned2 = nullptr;               // shape path: pinned host slots for inflated PNG scanlines
    size_t h_pinned2_bytes = 0;
};
void shape_release_dev(DevState &ds);

void set_tls_error(const std::string &msg);

// Every exported function runs its body through this: "nothing aborts or throws across the ABI" (include/cdsgpu.h).  A C++
// exception (std::bad_alloc from a vector sized by caller input, std::length_error, ...) would otherwise unwind through the C
// boundary and, in the Java binding, through FFM / JNI frames.  Locks taken inside the body are released by the unwinding.
template <class F>
inline cds_status abi_guard(const char *name, F &&body) noexcept
{
    try {
        return body();
    } catch (const std::bad_alloc &) {
        try { set_tls_error(std::string(name) + ": out of host memory"); } catch (...) {}
        return CDS_ERR_OOM;
    } catch (const std::exception &e) {
        try { set_tls_error(std::string(name) + ": " + e.what()); } catch (...) {}
        return CDS_ERR_CUDA;
    } catch (...) {
        try { set_tls_error(std::string(name) + ": unknown C++ exception"); } catch (...) {}
        return CDS_ERR_CUDA;
    }
}

}  // namespace cds

struct cds_ctx {
    std::vector<cds::DevState> devs;
    mutable std::recursive_mutex mu;
    mutable std::string err;
    cds_search_stats stats{};
    int64_t shape_inflate_window = 0;   // cds_ctx_set_option("shape_inflate_window"): most targets per window of cds_shape_score_pairs_files with device inflate (0 = 2048)
    int device_inflate = 1;       // cds_ctx_set_option("device_inflate"): 1 = gradient PNG files are inflated on the device (cds_inflate.cu), 0 = by host threads,
                                  // 2 = on the device, and every odd image is treated as refused (exercises the zlib fallback in tests)
    bool wide_lists = false;   // cds_ctx_set_option("wide_lists"): mask sets prepared from now on get interval-carrying word lists even when palettes would do
    int match_kernel = 0;      // cds_ctx_set_option("match_kernel"): 0 automatic, 1 candidate, 2 band, 3 gather
    int resident_occupancy = 1;   // cds_ctx_set_option("resident_occupancy"): 0 = always build occupancy bitmaps per target chunk
    int64_t stream_chunk = 256;   // cds_ctx_set_option("stream_chunk"): targets per chunk of cds_search_stream_rgb
    int fused_ingest = 1;         // cds_ctx_set_option("fused_ingest"): 1 = TIFF strips go straight to code words (tiff_encode_kernel), 0 = decode to RGB, then encode
    int64_t stream_chunk_bytes = 0xC0000000ll;   // cds_ctx_set_option("stream_chunk_bytes"): most file bytes per chunk (the strip table addresses them with 32 bits)
    int64_t stream_chunk_tiff = 4096;   // cds_ctx_set_option("stream_chunk_tiff"): targets per chunk of cds_search_stream_tiff
    int64_t best_list_bytes = (int64_t) 1 << 30;   // cds_ctx_set_option("best_list_bytes"): per-device list of passing pairs of the *_best_matches searches

    cds_status fail(cds_status code, const std::string &msg) const;
    cds_status check(cudaError_t e, const char *what) const;
    cds_status ensure_staging(cds::DevState &d, size_t bytes);
    cds_status ensure_pinned(cds::DevState &d, size_t bytes);
    cds_status ensure_scratch(cds::DevState &d, int slot, size_t bytes, void **out);
    cds_status ensure_match_scratch(cds::DevState &d);
    cds_status class_table_on(cds::DevState &d, double tol, const cds_class_interval **out);
};

struct cds_library {
    cds_ctx *ctx = nullptr;
    cds::PlaneGeom g{};
    int64_t capacity = 0;
    int64_t size = 0;
    int baked_threshold = 0;
    struct Shard {
        uint32_t *planes = nullptr;
        int64_t cap_local = 0;
        uint32_t *occ = nullptr;        // occupancy bitmaps [cap_local][tile rows][sectors + 1][bpitch] (cds_kernels.cuh), built on demand
        uint32_t *valid = nullptr;      // its scratch
        int64_t occ_done = 0;           // local targets covered by `occ`
    };
    int bpitch = 0;
    int occ_threshold = 0, occ_rings = -1;   // parameters `occ` was built for
    bool occ_on_the_fly = false;             // the bitmaps do not fit next to the planes: searches build them per target chunk
    std::vector<Shard> shards;

    int n_dev() const { return (int) shards.size(); }
    // block-cyclic mapping global <-> (device, local)
    void locate(int64_t gidx, int &dev, int64_t &local) const {
        int64_t blk = gidx / cds::kLibBlock;
        dev = (int) (blk % n_dev());
        local = (blk / n_dev()) * cds::kLibBlock + gidx % cds::kLibBlock;
    }
    int64_t global_of(int dev, int64_t local) const {
        int64_t blk_local = local / cds::kLibBlock;
        return (blk_local * n_dev() + dev) * cds::kLibBlock + local % cds::kLibBlock;
    }
    int64_t local_size(int dev) const;   // number of targets currently on `dev`
    cds_status bake(int threshold);      // make the below-threshold flags match `threshold`
    cds_status ensure_occupancy(int rings);   // occupancy bitmap for the baked threshold and this shift set, all devices
};

struct cds_maskset {
    cds_ctx *ctx = nullptr;
    int W = 0, H = 0;
    cds_pixparams params{};
    cds::ShiftSet shifts{};
    cds::RectSet rects{};
    std::vector<int32_t> sizes;          // getQuerySize() per mask
    // Growable device arenas, one set per device (identical contents: masks are replicated).  Records, colour classes and
    // compact records of all masks are contiguous in the order the masks were added; rowstart is [M][H+1].
    struct Arena { void *p = nullptr; size_t cap = 0, used = 0; };     // bytes
    struct DevStore { Arena records, classes, crec, rowstart; };
    std::vector<DevStore> store;                       // per device
    std::vector<uint64_t> rec_offset;                  // [M] index of each mask's first record inside the arenas
    std::vector<cds::MaskDesc *> d_descs;              // per device, rebuilt when dirty
    std::vector<cds::PaletteGroup *> d_groups;         // per device, one per CDS_PALETTE_GROUP masks
    std::vector<uint2 *> d_palettes;                   // per device, [n_groups][CDS_PALETTE_SIZE]
    std::vector<uint32_t *> d_words;                   // per device, word-list entries of all groups followed by their palette references (cds_cand.cuh)
    std::vector<uint32_t *> d_wstart;                  // per device, per-mask offsets and per-group row starts of the word lists
    int n_compact_groups = 0;                          // groups whose colour classes fit a shared-memory palette
    std::vector<int32_t> n_pal;                        // per group, its palette's size (0 without a palette); the same on every device
    bool wide_lpal = false;                            // the word lists carry intervals instead of palette references (cds_cand.cuh: WIDE)
    bool words_built = false;                          // the candidate kernel's word lists exist on every device
    bool descs_dirty = true;
    cds_status sync_descs();
};


namespace cds {
// What a match kernel needs to know about a run of device-resident targets (a library shard or one streamed chunk).
struct TargetView {
    const uint32_t *planes = nullptr;   // code planes, PlaneGeom layout
    const uint32_t *occ = nullptr;      // occupancy bitmap for the mask set's shift set and the baked threshold
    PlaneGeom g{};
    int bpitch = 0;
    int64_t n = 0;                      // targets
    bool occ_ready = false;
    bool bands = false;                 // the occupancy carries its rank-band bytes (cds_kernels.cuh): the library's resident bitmaps only
};
// Picks and launches the match kernel for masks [m0, m0 + mc) of `ms` against `tv` on `stream`; ev0 / ev1 (may be null) are
// recorded around it.  d_scores[(m - m0) * tv.n + t] = score word.
cds_status launch_match_view(cds_ctx *ctx, const cds_maskset *ms, const TargetView &tv, int d, int m0, int mc, int32_t *d_scores,
                             cudaStream_t stream, cudaEvent_t ev0, cudaEvent_t ev1);
bool batched_kernel_supported(int xy_shift, const PlaneGeom &g);
int choose_pitch(int W);
// smallest score in [1, P] with ColorMIPSearch.isMatch true; P + 1 when none
int32_t min_matching_score(int32_t P, double pct_positive_pixels);
// cds_search_topk over a resident library with occupancy bitmaps built per target chunk (cds_stream.cu)
cds_status search_library_chunked(cds_ctx *ctx, const cds_maskset *ms, cds_library *lib, int32_t k, double pct_positive_pixels,
                                  int32_t *out_score, int64_t *out_target, uint8_t *out_mirrored, int32_t *out_count);

// Appends n images at consecutive global indices; `src` fills the device staging buffer with the RGB pixels of images
// [i0, i0 + cnt) of the call (an H2D copy or a generator kernel) on ds.stream.
cds_status library_append(cds_library *lib, int64_t n,
                          const std::function<cds_status(DevState &, int64_t i0, int64_t cnt, uint8_t *d_rgb)> &src,
                          int64_t *first_index);
// one chunk of a search over host targets (cds_stream.cu)
struct StreamChunk { int d; int64_t first, cnt; };
std::vector<StreamChunk> stream_chunk_plan(int D, int64_t n_targets, int64_t chunk, const int64_t *offsets, uint64_t byte_cap);
// masks per chunk of maskset_append (and therefore the most consecutive files a TIFF source has to stage at once)
inline int maskset_append_chunk(int n)
{
    static const int forced = std::getenv("CDSGPU_MASK_CHUNK") ? std::atoi(std::getenv("CDSGPU_MASK_CHUNK")) : 0;      // tuning aid
    if (forced > 0) return forced;
    return n <= 64 ? 64 : 256;
}
// Appends n masks whose pixels `fill` puts into device staging memory (cds_api.cu).
cds_status maskset_append(cds_maskset *ms, int32_t n, int32_t *mask_size_out,
                          const std::function<cds_status(int i0, int cnt, uint8_t *stage, cudaStream_t stream)> &fill);
}  // namespace cds

#endif

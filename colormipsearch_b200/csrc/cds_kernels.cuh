// cds_kernels.cuh -- launch wrappers of the CUDA kernels (implemented in the .cu files of this directory).
#ifndef CDS_KERNELS_CUH
#define CDS_KERNELS_CUH

#include <cuda_runtime.h>
#include <stdint.h>
#include "cds_common.h"

namespace cds {

// Geometry of the encoded library planes in HBM (all in 32-bit words).
//   plane t, image row y (0 <= y < H), column x  ->  base[(guard + t * (H + guard) + y) * pitch + x]
// Every row has pitch - W >= CDS_MIN_PAD_COLS trailing pad words; `guard` pad rows separate consecutive planes and
// precede the first one, so a band of rows [y0 - s, y1 + s) of any plane is ONE contiguous, 16-byte aligned span that
// already contains the out-of-image pixels as never-matching pad words.
struct PlaneGeom {
    int W, H, pitch, guard;
    __host__ __device__ size_t plane_stride() const { return (size_t) (H + guard) * pitch; }
    __host__ __device__ size_t total_words(int64_t capacity) const { return ((size_t) capacity * (H + guard) + guard) * pitch; }
    __host__ __device__ size_t row_offset(int64_t t, int y) const { return ((size_t) guard + (size_t) t * (H + guard) + y) * pitch; }
};

struct RectSet {
    int n;
    int x0[8], y0[8], x1[8], y1[8];
};

// Per-mask descriptor on the device.
struct MaskDesc {
    const cds_mask_record *records;   // P records, ascending pixel index
    const uint32_t *rowstart;         // H + 1 entries: records of image row y are [rowstart[y], rowstart[y+1])
    const uint32_t *crec;             // P compact records (cds_common.h) or nullptr when the mask's palette group is wide
    const uint32_t *classes;          // P colour classes (sector * CDS_NUM_RANKS + rank, or CDS_CLASS_NONE_INDEX)
    const uint32_t *wstart;           // H + 1 entries: offset of this mask's entries inside its group's run of each row (cds_cand.cuh)
    int P;
    int pad;
};

// One palette group = CDS_PALETTE_GROUP consecutive masks.
struct PaletteGroup {
    const uint2 *palette;             // n_pal entries, or nullptr: the group uses the 16-byte records
    const uint4 *words;               // base of the word lists of the candidate kernel (cds_cand.cuh), or nullptr
    const uint32_t *gstart;           // H + 1 entries: this group's entries of image row y are words[gstart[y] .. gstart[y+1])
    const uint16_t *lpal;             // palette references of the entries' set bits (cds_cand.cuh)
    const uint32_t *tocc;             // occupancy word of every 32nd entry of `words` (cds_cand.cuh)
    int n_pal;
    int pad;
};

struct ShiftSet {
    int n;                            // offsets per orientation
    int mirror;
    int8_t dx[CDS_MAX_SHIFT_OFFSETS];
    int8_t dy[CDS_MAX_SHIFT_OFFSETS];
};

// Device scratch of the batched match kernels, owned by one context's device state (two contexts on one device must not share it):
// the work-item counter of the persistent grids and the candidate kernel's match counters.
struct MatchScratch {
    unsigned long long *work_counter = nullptr;
    int *acc = nullptr;                       // kMatchAccBytes, zero between launches
};
constexpr size_t kMatchAccBytes = (size_t) 256 * CDS_PALETTE_GROUP * ((CDS_MAX_VARIANTS + 3) / 4 * 4) * sizeof(int);   // [<= 256 CTAs][masks of a group][variants, padded to 16 bytes]

// score word written by the match kernels: matching pixels | mirrored << 30
#define CDS_SCORE_MIRROR_BIT 0x40000000

void launch_fill_words(uint32_t *p, size_t n, uint32_t v, cudaStream_t s);
// `valid` (optional): chunk-relative scratch [n][H][sectors][occupancy_valid_pitch(W)]; the encoder then also writes the per-sector
// "can match" bits of every row, and launch_occupancy can be called with valid_ready = true (no second pass over the planes).
void launch_encode_rgb(const uint8_t *rgb, int64_t n, uint32_t *planes, PlaneGeom g, int64_t first_slot,
                       const uint16_t *rank_tab, int data_threshold, cudaStream_t s, uint32_t *valid = nullptr);
void launch_rebake(uint32_t *planes, size_t n_words, int data_threshold, cudaStream_t s);
void launch_encode_colors(const uint8_t *rgb, int64_t n, const uint16_t *rank_tab, int data_threshold, uint32_t *codes, cudaStream_t s);

// Occupancy bitmaps of the library, in TILES of 8 x 4 pixels: bit (y % 4) * 8 + (x % 8) of tile word (y / 4, x / 8).  Per target
// and tile row there are CDS_NUM_SECTORS + 1 rows of `tp` tile words each (occupancy_row_pitch(tp) words per tile row): bit (x, y)
// of sector row s is set when at least one of the pixels (x + dx, y + dy), (dx, dy) in the shift set of `rings` (0: centre only,
// 1: {-2,0,2}^2, 2: additionally {-4,0,4}^2), is inside the image, above the baked threshold and of colour sector s; the last
// row is the OR of the sector rows.  A mask pixel can only match target pixels of the sector of one of its (at most two) rank
// intervals, so a clear bit in that sector's row means "cannot match in any shifted variant"; the shift set being symmetric, the
// bit of the mirrored position covers the mirrored variants.  (Tiles rather than 32 x 1 strips because a neurite a few pixels
// wide fills a compact tile much better than a strip: 1.8 x fewer non-empty mask words to scan, cds_cand.cuh.)
// The bitmaps must be zero before the first launch_occupancy (bytes of rows beyond the image are never written).
// `valid_scratch` holds scratch_targets * H * CDS_NUM_SECTORS * occupancy_valid_pitch(W) words (row layout, one bit per pixel).
__host__ __device__ inline int occupancy_valid_pitch(int W) { return (((W + 31) / 32) + 3) / 4 * 4; }
__host__ __device__ inline int occupancy_tile_pitch(int W) { return (((W + 7) / 8) + 3) / 4 * 4; }
__host__ __device__ inline int occupancy_tile_rows(int H) { return (H + 3) / 4; }
// A tile row is laid out as
//   [sector rows: CDS_NUM_SECTORS * tp words][non-empty bits: occupancy_nz_words(tp)][rank-band bytes: occupancy_band_words(tp)][OR row: tp]
// The first three parts (occupancy_stage_pitch(tp) words) are what the candidate kernel stages per tile row; the word lists index
// them (tile row * occupancy_stage_pitch + sector * tp + tile column).  The OR row, read by the band kernel only, comes last.
//   * non-empty bits: one BIT per sector tile word, "this word is not empty" (bit i = word i of the tile row, i < CDS_NUM_SECTORS * tp).
//     The candidate kernel's ticket tests read these.
//   * rank-band bytes: byte i (bits 8 (i % 4) .. 8 (i % 4) + 7 of word i / 4) belongs to sector tile word i and has bit b set when
//     one of the target pixels that can set that word's bits has rank band b (occupancy_rank_band): a pixel of the word's sector,
//     inside the image, above the baked threshold, in the rectangle [8 tx - S, 8 tx + 7 + S] x [4 ty - S, 4 ty + 3 + S] (S = xyShift).
//     That rectangle is exactly the union of the shifted tile for xyShift 2 and 4 except in a last tile row that holds a single image
//     row, where it is a superset; for xyShift 0 it is the tile itself.  Written by launch_occupancy with `bands` -- for the library's resident
//     bitmaps, which serve every later search.  Bitmaps built per streamed chunk serve one search: there the bytes cost more time than
//     the filter saves (DESIGN.md §4.1, v21), so they are not built and the candidate kernel runs without the filter.
__host__ __device__ inline int occupancy_nz_words(int tp) { return ((CDS_NUM_SECTORS * tp + 31) / 32 + 3) / 4 * 4; }
__host__ __device__ inline int occupancy_band_words(int tp) { return ((CDS_NUM_SECTORS * tp + 3) / 4 + 3) / 4 * 4; }
__host__ __device__ inline int occupancy_nz_offset(int tp) { return CDS_NUM_SECTORS * tp; }
__host__ __device__ inline int occupancy_band_offset(int tp) { return CDS_NUM_SECTORS * tp + occupancy_nz_words(tp); }
__host__ __device__ inline int occupancy_stage_pitch(int tp) { return occupancy_band_offset(tp) + occupancy_band_words(tp); }
__host__ __device__ inline int occupancy_any_offset(int tp) { return occupancy_stage_pitch(tp); }
__host__ __device__ inline int occupancy_row_pitch(int tp) { return occupancy_stage_pitch(tp) + tp; }
__host__ __device__ inline size_t occupancy_target_words(int W, int H) { return (size_t) occupancy_tile_rows(H) * occupancy_row_pitch(occupancy_tile_pitch(W)); }
// Rank bands: every sector's CDS_NUM_RANKS ranks cut into CDS_RANK_BANDS equal runs.  A fixed table, so that the target tiles' bytes and
// the mask entries' bytes (cds_cand.cu) agree without any data-dependent state.  One bit per band: at most 8.
#define CDS_RANK_BANDS 8
__host__ __device__ inline uint32_t occupancy_rank_band(uint32_t rank) { return rank * CDS_RANK_BANDS / CDS_NUM_RANKS; }
int &occupancy_kernel_version();      // cds_ctx_set_option("occupancy_kernel")
// `bands`: also the rank-band bytes (from the valid bits and the ranks in the code planes, which must then be given).
void launch_occupancy(const uint32_t *planes, PlaneGeom g, int64_t t0, int64_t n, int rings, int tp,
                      uint32_t *valid_scratch, int64_t scratch_targets, uint32_t *occ, cudaStream_t s, bool valid_ready = false,
                      bool bands = false);

void launch_mask_count_rows(const uint8_t *rgb, int n_masks, int W, int H, int threshold, RectSet rects,
                            uint32_t *rowcount, cudaStream_t s);
void launch_mask_scan_rows(uint32_t *rowcount, int n_masks, int H, int32_t *sizes, cudaStream_t s);
void launch_mask_write_records(const uint8_t *rgb, int n_masks, int W, int H, int threshold, RectSet rects,
                               const uint32_t *rowstart, const uint64_t *rec_offset, const uint16_t *rank_tab,
                               const cds_class_interval *class_tab, cds_mask_record *records, uint32_t *classes, cudaStream_t s);

// Palette construction for n_groups groups of consecutive masks (descs[g * CDS_PALETTE_GROUP ...]); `classes` pointers come
// with the descriptors.  flags / pidx: scratch [n_groups][CDS_NUM_CLASSES + 1].
struct MaskClassRef { const uint32_t *classes; const cds_mask_record *records; uint32_t *crec; int P; int pad; };
void launch_palette_mark(const MaskClassRef *masks, int n_masks, uint32_t *flags, cudaStream_t s);
void launch_palette_scan(const uint32_t *flags, int n_groups, uint32_t *pidx, int32_t *n_pal, cudaStream_t s);
void launch_palette_fill(const uint32_t *flags, const uint32_t *pidx, int n_groups, const cds_class_interval *class_tab,
                         uint2 *palettes /* [n_groups][CDS_PALETTE_SIZE] */, cudaStream_t s);
void launch_palette_records(const MaskClassRef *masks, int n_masks, const uint32_t *pidx, const int32_t *n_pal, cudaStream_t s);

void launch_pixelmatch_gather(const MaskDesc *masks, int n_masks, const uint32_t *planes, PlaneGeom g,
                              int64_t n_targets, ShiftSet shifts, int32_t *scores /* [n_masks][n_targets] */,
                              cudaStream_t s);

}  // namespace cds
#endif

// cds_cand.cuh -- the candidate kernel: batched pixel match driven by 32-pixel mask words (the hot path at scale).
#ifndef CDS_CAND_CUH
#define CDS_CAND_CUH

#include "cds_kernels.cuh"

#include <algorithm>

namespace cds {

// WORD LISTS of a mask group (built once per mask set, per device).
// A mask pixel can only match target pixels whose colour sector is the sector of one of its (at most two) rank intervals: its
// own sector (interval 1) and, near a sector boundary, one neighbouring sector (interval 2).  Per mask, orientation and
// sector the kernel keeps a bitmap in TARGET coordinates (orientation 0: pixel (x, y); orientation 1, only when the mask set
// mirrors: pixel (W-1-x, y)) of the pixels with an interval in that sector, cut into TILES of 8 x 4 pixels like the library's
// occupancy bitmaps (bit (y % 4) * 8 + (x % 8) of tile (y / 4, x / 8)) and stored as its non-zero 32-bit tile words.  The
// words of the CDS_PALETTE_GROUP masks of a group form ONE list ordered by tile row (then sector, tile column -- the order of the
// occupancy words --, then whatever) with a row-start table gstart[tile rows + 1], so the entries that concern a band of image rows are one contiguous
// range that is cut into equal tickets regardless of mask boundaries.  One 16-byte entry per word:
//     bits : the tile word
//     occ  : bits 0..23: index of the matching occupancy word inside a target's bitmaps: tile row * occupancy_stage_pitch + sector * pitch
//            + tile column (< 2^20 at W <= 2048, H <= 1024); bits 24..31: the word's rank-band byte, the OR over its set bits of the
//            rank bands (occupancy_rank_band) that the pixel's interval in this list's sector touches.  Readers mask the index with
//            kWordOccMask.
//     lrec : index into the group's `lpal` array of the palette reference of the word's LOWEST set bit; set bit b has
//            lpal[lrec + popc(bits below b)] = palette index | 0x8000 when the pixel is in this list through its interval 2
//            WIDE lists (a group of the set has more colour classes than a palette holds, e.g. brightness-scaled LM images used
//            as masks): `lpal` has 32 bits per set bit and holds the packed interval of this list's sector itself
//            (lo | len << 18 like a palette word); the kernel's WIDE instantiation then needs no palette.
//     meta : tile row | tile column << 8 | orientation << 16 | sector << 17 | mask index inside the group << 22 (10 bits)   (H <= 1024, W <= 2048)
// The scan reads whole entries (16 bytes, one 128-bit load) and uses {bits, occ}; {lrec, meta} travel with the words that have candidates.
// ANDing `bits` with the library's occupancy word of the same (tile row, sector, tile column) leaves exactly the mask pixels
// that can match in some shifted variant of that orientation -- 32 pixels per instruction -- and an evaluation tests ONE
// interval: the two lists of a boundary pixel partition its matches by target sector, so nothing is counted twice.
constexpr int kWordMetaColShift = 8;
constexpr int kWordMetaOrientBit = 16;
constexpr int kWordMetaSectorShift = 17;
constexpr int kWordMetaMaskShift = 22;
constexpr uint32_t kWordOccMask = (1u << 24) - 1u;
constexpr int kWordBandShift = 24;

bool cand_kernel_supported(int xy_shift, const PlaneGeom &g);

// Palette entries a launch stages in shared memory: `pal_entries` = the largest palette of the launch's groups plus the idle entry that
// idle lanes read (0 for WIDE lists, which read no palette), rounded up to 16.  The idle entry is the last staged one.
inline int cand_staged_palette(int pal_entries) { return pal_entries <= 0 ? 0 : std::min((pal_entries + 15) / 16 * 16, CDS_PALETTE_SIZE); }
// What a launch at this geometry and palette size runs with: consumer warps, band height, stages in flight and dynamic shared memory
// (ok = false: no configuration fits).  Host only; tests read it through cds_debug_cand_config.
struct CandShape {
    int warps, rows_per_band, n_stages;
    size_t smem_bytes;
    bool ok;
};
CandShape cand_launch_shape(int xy_shift, const PlaneGeom &g, int pal_entries);

// Tuning knobs of the candidate kernel (process-wide; defaults from the environment, changed through cds_ctx_set_option
// "cand_wait_mode" / "cand_l2_hint" / "cand_warps" so that one process can sweep them).
struct CandTuning {
    int wait_mode;      // how a consumer warp waits for a band: 0 polls try_wait, 1 try_wait with a suspend-time hint, n >= 2 test_wait + nanosleep(n ns)
    int l2_hint;        // 1: bulk copies of the streamed planes are evict-first, loads of the group's lists evict-last
    int warps;          // consumer warps per CTA (31, 28, 24 or 16)
    int stages;         // band stages in flight (2 .. 4); more stages mean shorter bands
    int max_rows;       // upper bound of the band height (0: as tall as shared memory allows)
};
CandTuning &cand_tuning();

// Construction, in this order (class_tab: the device interval table of the mask set's zTolerance):
//   launch_words_count      wcount[m][ty] / bcount[m][ty] = entries / set bits of (mask m, tile row ty); arrays are [.][tile rows + 1]
//   launch_words_group_rows (once per array, H = tile rows) count[m][ty] -> offset of mask m inside its group's run; grow[g][ty] = run length
//   (host) gstart / bstart = exclusive scans of the two grow arrays over (group, row), absolute indices; [g][H] = end of the group
//   launch_words_fill       writes entries and palette references; masks[m].wstart must point at wcount[m], boff at bcount
void launch_words_count(const MaskDesc *masks, int n_masks, int W, int H, bool mirror, const cds_class_interval *class_tab,
                        uint32_t *wcount, uint32_t *bcount, cudaStream_t s);
void launch_words_group_rows(uint32_t *count, int n_masks, int H, uint32_t *grow, cudaStream_t s);
void launch_words_fill(const MaskDesc *masks, int n_masks, int W, int H, bool mirror, const cds_class_interval *class_tab,
                       const uint32_t *gstart, const uint32_t *bstart, const uint32_t *boff, uint4 *words, uint16_t *lpal, cudaStream_t s,
                       bool wide_lpal = false);

// Reorders every tile row's entries by occupancy word (`occ`), i.e. by (sector, tile column): afterwards the entries that meet one
// target tile are neighbours, and the kernel skips the tickets whose occupancy words are all empty.  `tables` = scratch of
// 2 * n_groups * words_bucket_count(W, H) words; `sorted` receives the entries (same size as `words`, must not alias it).
inline size_t words_bucket_count(int W, int H) { return (size_t) occupancy_tile_rows(H) * occupancy_stage_pitch(occupancy_tile_pitch(W)); }
void launch_words_bucket_sort(const uint4 *words, const uint32_t *gstart, int n_groups, int W, int H, uint32_t *tables, uint4 *sorted, cudaStream_t s);
// PaletteGroup::tocc of the SORTED list: the occupancy word of every 32nd entry, words_tocc_count(n_entries) words.
inline uint32_t words_tocc_count(uint32_t n_entries) { return n_entries / 32 + 2; }
void launch_words_tocc(const uint4 *words, uint32_t n_entries, uint32_t *tocc, cudaStream_t s);

// Same contract as launch_pixelmatch_band (cds_band.cuh); every group needs a palette and its word lists
// (PaletteGroup::palette / words / gstart / lpal).  `pal_entries`: the largest n_pal + 1 over the launch's groups (0 for WIDE lists).
// `band_bytes`: the occupancy carries its rank-band bytes (cds_kernels.cuh), and the kernel filters words with them.
int launch_pixelmatch_cand(const MaskDesc *masks, int n_masks, const uint32_t *planes, PlaneGeom g, int64_t n_targets,
                           const uint32_t *occ, int bpitch, const PaletteGroup *groups, int xy_shift, bool mirror,
                           int32_t *scores, const MatchScratch &scratch, cudaStream_t s, bool wide_lpal, bool band_bytes, int pal_entries);

}  // namespace cds
#endif

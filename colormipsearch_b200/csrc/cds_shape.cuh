// cds_shape.cuh -- what the shape score's two pair kernels share (shape_pair_kernel in cds_shape.cu for the batched call,
// shape_pair_batch_kernel in cds_shape_pairq.cu for the single-pair queue): the prepared masks, the per-pixel gap arithmetic,
// the high-expression count and the mirror rule, so that the formula exists once.
#pragma once

#include <vector>

#include "cds_runtime.h"

namespace cds {

// one prepared mask on one device
struct ShapeMaskDesc {
    const uint32_t *gap_list;    // x | y << 11 | (slice(Q) - 1) << 21 | QM << 29 | keep_normal << 30 | keep_mirrored << 31
    const uint32_t *he_n, *he_m; // high-expression bitmap and its row-mirrored copy, [H][bpitch]
    int n_gap;
    int pad;
};

// PIXEL_GAP_OP (API/cds/Shape2DMatchColorDepthSearchAlgorithm.java:30-37) for one entry of a mask's gap list, in both orientations of
// the query: the gap counts only above 3, the gradient term carries the query mask QM, and the mirrored query reads the gradient at the
// mirrored column while the zgap image is sampled at the query's own pixel.  zs / gr: the target's slice and gradient planes [H][W].
__device__ __forceinline__ void shape_gap_entry(uint32_t e, const uint16_t *zs, const uint16_t *gr, int W, int mirror, long long &gap_n,
                                                long long &gap_m)
{
    const int x = (int) (e & 0x7FFu), y = (int) ((e >> 11) & 0x3FFu);
    const int qs = (int) ((e >> 21) & 0xFFu) + 1;
    const int qm = (int) ((e >> 29) & 1u);
    const size_t rowoff = (size_t) y * W;
    const int z = zs[rowoff + x];                            // the zgap image is sampled at the query's own pixel in both orientations
    int big = 0;
    if (z != 0) {                                            // PIXEL_GAP_OP :30-37
        const int pxGapSlice = abs(qs - z);
        if (40 <= pxGapSlice - 40) big = pxGapSlice - 40;
    }
    if (e & 0x40000000u) {
        const int gap = big ? big : qm * (int) gr[rowoff + x];
        if (gap > 3) gap_n += gap;
    }
    if (mirror && (e & 0x80000000u)) {
        const int gap = big ? big : qm * (int) gr[rowoff + (W - 1 - x)];   // the gradient is NOT mirrored with the query :222
        if (gap > 3) gap_m += gap;
    }
}

// word i of the high-expression area: the mask's bitmaps AND the target's signal bitmap ts
__device__ __forceinline__ void shape_he_word(const ShapeMaskDesc &md, const uint32_t *ts, int i, int mirror, long long &he_n, long long &he_m)
{
    const uint32_t tw = ts[i];
    he_n += __popc(__ldg(md.he_n + i) & tw);
    if (mirror) he_m += __popc(__ldg(md.he_m + i) & tw);
}

// tot = {gap, mirrored gap, high-expression area, mirrored area} -> the pair's (gap, area); returns 1 when the mirrored query wins:
// ShapeMatchScore.getScore narrows calculate2DShapeScore to int; mirrored wins when strictly smaller (:181)
__device__ __forceinline__ int shape_pick(const long long tot[4], int mirror, long long &g, long long &h)
{
    g = tot[0]; h = tot[2];
    if (mirror) {
        const int s0 = (int) (tot[0] + tot[2] / 3);
        const int s1 = (int) (tot[1] + tot[3] / 3);
        if (s1 < s0) { g = tot[1]; h = tot[3]; return 1; }
    }
    return 0;
}

}  // namespace cds

// ------------------------------------------------------------------------------------------------------------------ prepared masks
struct cds_shape_maskset {
    cds_ctx *ctx = nullptr;
    int W = 0, H = 0, bpitch = 0;
    int query_threshold = 0, mirror = 0;
    cds::RectSet rects{};
    uint32_t *d_roi_bits = nullptr;                  // label-cleared ROI bitmap on device 0 (where masks are prepared), or nullptr
    int n_masks = 0;
    // per device: the masks' descriptors (device-local pointers), the blocks that hold their lists and bitmaps
    struct Dev {
        std::vector<cds::ShapeMaskDesc> h_descs;
        std::vector<void *> blocks;
        cds::ShapeMaskDesc *d_descs = nullptr;
        size_t d_descs_cap = 0;
        bool dirty = true;
    };
    std::vector<Dev> dev;
};

namespace cds {

// The target side of n pairs on device ds, as the scoring path derives it: zslice [n][H][W] = slice numbers of the thresholded zgap
// images -- the given ones (zgap != nullptr, target_planes_kernel) or maxFilter(10)(mask(threshold)(clearLabels(target))) derived on
// the device (shape_target_derive_kernel) --, tsig [n][H][bpitch] = the targets' "above threshold outside labels" bitmaps.
void launch_shape_target_planes(const cds_shape_maskset *sms, const DevState &ds, const uint8_t *target, const uint8_t *zgap, int64_t n,
                                uint16_t *zslice, uint32_t *tsig, cudaStream_t s);

}  // namespace cds

// cds_shape.cu -- 2D shape (gradient area gap) scoring on the device.
//
// Reference semantics (API/ = colormipsearch-api/src/main/java/org/janelia/colormipsearch/):
//   per-mask preparation : ColorDepthSearchAlgorithmProviderFactory.createShapeMatchCDSAlgorithmProvider, API/cds/...ProviderFactory.java:76-127
//   max filter           : ImageTransformation.unsafeMaxFilter / makeLineRadii, API/imageprocessing/ImageTransformation.java:353-572
//   gray / signal / mask : API/imageprocessing/ColorTransformation.java:29-54, 97-160
//   slice numbers        : GradientAreaGapUtils.calculateSliceGap / findSliceNumber(InLUT), API/cds/GradientAreaGapUtils.java:18-197
//   pair score           : Shape2DMatchColorDepthSearchAlgorithm.calculateMatchingScore / calculateNegativeScores / PIXEL_GAP_OP,
//                          API/cds/Shape2DMatchColorDepthSearchAlgorithm.java:26-42, 150-245
//
// B200 formulation.  PIXEL_GAP_OP is zero wherever the (label-cleared, ROI-masked) query pixel is black -- its "queryMask * gradient"
// term needs gray(query) > 2 -- so the gradient-area gap is a sum over the query's NON-BLACK pixels only (~1-3 % of the image).
// Per mask the devices keep (a) that pixel list with the query's slice number folded in, (b) the high-expression mask and its
// row-mirrored copy as bitmaps.  Per target a device keeps, for as long as the target's window is being scored, the slice-number
// plane of the thresholded zgap image, the gradient plane and the "above threshold outside labels" bitmap.  One CTA scores one
// (mask, target) pair in both orientations: a gather over the pixel list for the gaps, and an AND + POPC sweep over the bitmaps for
// the high-expression area.
//
// What is new against the first version of this file (profiles/r01_shape_launches.csv: the u8 disc max filter took 65 % of the
// device time at 1.8 % of the HBM peak, the slice planes 23 %, the pair kernel 3 %):
//   * the zgap image is never materialised.  shape_target_derive_kernel stages a tile of the thresholded, label-cleared target as
//     16-bit lanes (two pixels per 32-bit word), dilates it with the ImageJ disc by a nested-rectangle (Horner) scheme whose only
//     arithmetic is the 3-input packed maximum VIMNMX3.U16x2, and turns the three channel maxima straight into a slice number.
//   * slice numbers come from a table [max/second channel pair][max][second] built once per device by the reference's own double
//     arithmetic (findSliceNumberInLUT), not from up to 56 double divisions per pixel.
//   * the mask side only ever needs ZERO / NON-ZERO facts about the r = 60 and r = 20 dilations, so it is binary morphology on
//     bitmaps (64 pixels per lane and instruction) instead of two u8 disc filters; masks are prepared in batches with one
//     device round trip per batch instead of two per mask.
//   * targets are processed in windows (device memory does not grow with the call) that are dealt out over ALL devices of the
//     context; the shape mask data is replicated like the pixel-match masks (SURVEY 8e: pairs go to the device that holds the target).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <memory>
#include <numeric>
#include <vector>

#include "cds_lut.h"
#include "cds_runtime.h"
#include "cds_shape.cuh"
#include "cds_tiff.h"

using namespace cds;

namespace cds {

// ------------------------------------------------------------------------------------------------------------------ slice numbers
__constant__ uint8_t c_shape_lut[256 * 3];

// findSliceNumberInLUT, API/cds/GradientAreaGapUtils.java:131-197 (IEEE double, no contraction: the file is built with --fmad=false)
__device__ int find_slice_in_lut(int lo, int hi, double colorRatio)
{
    int sliceNumber = 0;
    double mingapratio = 1000;
    for (int i = lo; i <= hi; i++) {
        const double colorR = c_shape_lut[3 * i], colorG = c_shape_lut[3 * i + 1], colorB = c_shape_lut[3 * i + 2];
        double lutRatio = 0;
        if (colorB > colorR && colorB > colorG) {
            if (colorR > colorG) lutRatio = colorR / colorB;
            else if (colorG > colorR) lutRatio = colorG / colorB;
        } else if (colorG > colorR && colorG > colorB) {
            if (colorR > colorB) lutRatio = colorR / colorG;
            else if (colorB > colorR) lutRatio = colorB / colorG;
        } else if (colorR > colorG && colorR > colorB) {
            if (colorG > colorB) lutRatio = colorG / colorR;
            else if (colorB > colorG) lutRatio = colorB / colorR;
        }
        if (lutRatio == colorRatio) return i + 1;
        const double gapratio = fabs(colorRatio - lutRatio);
        if (gapratio < mingapratio) { mingapratio = gapratio; sliceNumber = i + 1; }
    }
    return sliceNumber;
}

// The slice of a colour is a function of (which channel is the maximum, which is the second -- ties resolved by the >= order of
// calculateSliceGap :31-93 --, the two values): 6 x 256 x 256 entries, built once per device with the arithmetic above.
//   pair 0: R max, G second (LUT 171..212)   1: R, B (213..255)   2: G, R (128..170)   3: G, B (86..127)   4: B, R (0..29)   5: B, G (30..85)
constexpr int kSliceTabEntries = 6 * 65536;

__global__ void build_slice_table_kernel(uint16_t *__restrict__ tab)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kSliceTabEntries) return;
    const int pair = i >> 16, max1 = (i >> 8) & 255, max2 = i & 255;
    const int lo[6] = {171, 213, 128, 86, 0, 30}, hi[6] = {212, 255, 170, 127, 29, 85};
    int s = 0;
    if (max1 > 0 && max2 <= max1) s = find_slice_in_lut(lo[pair], hi[pair], (double) max2 / (double) max1);
    tab[i] = (uint16_t) s;
}

// first half of calculateSliceGap (:18-99) + findSliceNumber (:107-129).  0 for black.
__device__ __forceinline__ int slice_of(const uint16_t *__restrict__ tab, int red, int green, int blue)
{
    if ((red | green | blue) == 0) return 0;
    int max1, max2, pair;
    if (red >= green && red >= blue) {
        max1 = red;
        if (green >= blue) { max2 = green; pair = 0; } else { max2 = blue; pair = 1; }
    } else if (green >= red && green >= blue) {
        max1 = green;
        if (red >= blue) { max2 = red; pair = 2; } else { max2 = blue; pair = 3; }
    } else {
        max1 = blue;
        if (red >= green) { max2 = red; pair = 4; } else { max2 = green; pair = 5; }
    }
    return (int) __ldg(tab + ((pair << 16) | (max1 << 8) | max2));
}

__global__ void slice_numbers_kernel(const uint8_t *__restrict__ rgb, int64_t n, const uint16_t *__restrict__ tab, uint16_t *__restrict__ out)
{
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x)
        out[i] = (uint16_t) slice_of(tab, rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2]);
}

__device__ __forceinline__ bool shape_in_rects(const RectSet &r, int x, int y)
{
    bool in = false;
#pragma unroll
    for (int i = 0; i < 8; i++)
        if (i < r.n) in |= (x >= r.x0[i] && x < r.x1[i] && y >= r.y0[i] && y < r.y1[i]);
    return in;
}

// rgbToGrayNoGammaCorrection with maxGrayValue 255 (ColorTransformation.java:40-54, :103) in its exact integer form
// floor((2 (r + g + b) + 3) / 6): the double expression is never within 1/6 of an integer boundary (checked over ALL 2^24 colours
// against the oracle's double expression, tests/test_oracle_golden.py::test_gray_integer_form)
__device__ __forceinline__ int gray_of(int r, int g, int b) { return (r | g | b) == 0 ? 0 : (2 * (r + g + b) + 3) / 6; }

// ------------------------------------------------------------------------------------------------------------------ the ImageJ disc
// makeLineRadii, API/imageprocessing/ImageTransformation.java:549-572: rows dy = -k..k with half widths dxs[dy + k].
struct DiscSpec {
    int k;
    int dxs[121];      // half widths for dy = -k..k (k <= 60)
};

static DiscSpec make_disc(double radiusArg)
{
    DiscSpec d{};
    double radius;
    if (radiusArg >= 1.5 && radiusArg < 1.75) radius = 1.75;
    else if (radiusArg >= 2.5 && radiusArg < 2.85) radius = 2.85;
    else radius = radiusArg;
    const int r2 = (int) (radius * radius) + 1;
    const int k = (int) (std::sqrt(r2 + 1e-10));
    d.k = k;
    if (k > 60) return d;
    for (int y = -k; y <= k; y++) d.dxs[y + k] = (y == 0) ? k : (int) (std::sqrt(r2 - y * y + 1e-10));
    return d;
}

// The disc as a union of nested rectangles.  Its half widths never grow with |dy|, so with w_1 > w_2 > .. > w_n the distinct
// half widths and h_i the largest |dy| whose row is at least w_i wide, disc = U_i [-w_i, w_i] x [-h_i, h_i] (h grows as w shrinks).
// A max (or OR) over a rectangle is a horizontal max of half width w_i of the vertical max over |dy| <= h_i, and because both
// families are nested the whole union evaluates Horner-style:
//     X = 0;  for i = 1..n:  X = max(X, rows h_(i-1) < |dy| <= h_i);  X = hmax_(w_i - w_(i+1))(X)        (w_(n+1) = 0)
// i.e. every row of the window is read once (2k + 1 reads) and the horizontal work is w_1 = k single-pixel steps in total,
// whatever the number of rectangles.
struct DiscRings {
    int k, n;
    int8_t h[64];      // last |dy| of ring i
    int8_t d[64];      // horizontal steps after ring i
};

static DiscRings make_rings(const DiscSpec &disc)
{
    DiscRings r{};
    r.k = disc.k;
    int i = 0;
    for (int dy = 0; dy <= disc.k;) {
        const int w = disc.dxs[disc.k + dy];
        int last = dy;
        while (last + 1 <= disc.k && disc.dxs[disc.k + last + 1] == w) last++;
        const int wn = last + 1 <= disc.k ? disc.dxs[disc.k + last + 1] : 0;
        r.h[i] = (int8_t) last;
        r.d[i] = (int8_t) (w - wn);
        i++;
        dy = last + 1;
    }
    r.n = i;
    return r;
}

// ------------------------------------------------------------------------------------------------------------------ u8 max filter (generic radii)
// Kept for cds_make_zgap with radii beyond the fused kernel's halo (k > 16): one CTA produces a TR x TC tile of one channel from a
// sparse table of horizontal running maxima.  Not on the scoring path.
constexpr int kMfTR = 16, kMfTC = 64;

__global__ void __launch_bounds__(256) max_filter_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int W, int H, int nch,
                                                         DiscSpec disc, int nlev)
{
    extern __shared__ uint8_t s_lev[];               // [nlev][rows][cols]
    __shared__ int s_row_lev[121], s_row_off[121];
    const int k = disc.k;
    const int rows = kMfTR + 2 * k, cols = kMfTC + 2 * k;
    const int plane = rows * cols;
    const int x0 = blockIdx.x * kMfTC, y0 = blockIdx.y * kMfTR;
    const int img = blockIdx.z / nch, ch = blockIdx.z % nch;
    const uint8_t *s = src + (size_t) img * W * H * nch + ch;
    uint8_t *d = dst + (size_t) img * W * H * nch + ch;

    int nz = 0;
    for (int i = threadIdx.x; i < plane; i += blockDim.x) {
        const int r = i / cols, c = i % cols;
        const int x = x0 - k + c, y = y0 - k + r;
        uint8_t v = 0;
        if (x >= 0 && x < W && y >= 0 && y < H) v = s[((size_t) y * W + x) * nch];
        s_lev[i] = v;
        nz |= v;
    }
    for (int i = threadIdx.x; i < 2 * k + 1; i += blockDim.x) {
        const int L = 2 * disc.dxs[i] + 1;
        int j = 0;
        while ((2 << j) <= L) j++;
        s_row_lev[i] = j;
        s_row_off[i] = L - (1 << j);
    }
    const int any = __syncthreads_or(nz);
    if (!any) {
        for (int i = threadIdx.x; i < kMfTR * kMfTC; i += blockDim.x) {
            const int x = x0 + i % kMfTC, y = y0 + i / kMfTC;
            if (x < W && y < H) d[((size_t) y * W + x) * nch] = 0;
        }
        return;
    }
    for (int j = 1; j < nlev; j++) {
        const uint8_t *prev = s_lev + (size_t) (j - 1) * plane;
        uint8_t *cur = s_lev + (size_t) j * plane;
        const int step = 1 << (j - 1);
        for (int i = threadIdx.x; i < plane; i += blockDim.x) {
            const int c = i % cols;
            uint8_t v = prev[i];
            if (c + step < cols) v = max(v, prev[i + step]);
            cur[i] = v;
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < kMfTR * kMfTC; i += blockDim.x) {
        const int ox = i % kMfTC, oy = i / kMfTC;
        const int x = x0 + ox, y = y0 + oy;
        if (x >= W || y >= H) continue;
        int m = 0;
        for (int dy = -k; dy <= k; dy++) {
            const int w = disc.dxs[dy + k];
            const uint8_t *row = s_lev + (size_t) s_row_lev[dy + k] * plane + (size_t) (oy + k + dy) * cols + (ox + k - w);
            m = max(m, max((int) row[0], (int) row[s_row_off[dy + k]]));
        }
        d[((size_t) y * W + x) * nch] = (uint8_t) m;
    }
}

static bool launch_max_filter(const uint8_t *src, uint8_t *dst, int64_t n, int W, int H, int nch, const DiscSpec &disc, cudaStream_t s)
{
    if (disc.k > 60 || disc.k < 0) return false;
    int nlev = 1;
    while ((1 << nlev) <= 2 * disc.k + 1) nlev++;
    const size_t smem = (size_t) nlev * (kMfTR + 2 * disc.k) * (kMfTC + 2 * disc.k);
    cudaFuncSetAttribute(max_filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    for (int64_t i0 = 0; i0 < n; i0 += 8192) {
        const int64_t cnt = std::min<int64_t>(8192, n - i0);
        dim3 grid((W + kMfTC - 1) / kMfTC, (H + kMfTR - 1) / kMfTR, (unsigned) (cnt * nch));
        max_filter_kernel<<<grid, 256, smem, s>>>(src + (size_t) i0 * W * H * nch, dst + (size_t) i0 * W * H * nch, W, H, nch, disc, nlev);
    }
    return true;
}

// dst = clearRegion(src) then optionally mask(threshold): black inside label rectangles, black where every channel <= threshold
__global__ void clear_and_mask_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int64_t n, int W, int H, RectSet rects,
                                      int threshold, int apply_mask)
{
    const size_t total = (size_t) n * W * H;
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
        const int x = (int) (i % W), y = (int) ((i / W) % H);
        int r = src[3 * i], g = src[3 * i + 1], b = src[3 * i + 2];
        bool keep = !shape_in_rects(rects, x, y);
        if (apply_mask) keep = keep && (r > threshold || g > threshold || b > threshold);
        if (!keep) r = g = b = 0;
        dst[3 * i] = (uint8_t) r; dst[3 * i + 1] = (uint8_t) g; dst[3 * i + 2] = (uint8_t) b;
    }
}

// ------------------------------------------------------------------------------------------------------------------ target side, fused
// zslice(x, y) = slice number of mask(threshold)(maxFilter_r(mask(threshold)(clearLabels(target))))(x, y), tsig bit = clearLabels(target)
// above threshold -- Shape2DMatchColorDepthSearchAlgorithm.java:159-161 with the zgap image the reference's tests derive
// (Shape2DMatchColorDepthSearchAlgorithmTest.java:171-174) -- in one pass over the target's RGB bytes.
//
// A CTA produces kZgTH rows x kZgStrip columns.  The strip plus kZgHalo columns on either side (128 pixels) and the rows plus k
// above and below are staged per channel as u16 lanes, two pixels per word (pixel 2j in the low half of word j).  A warp then
// owns one output row at a time; lane l holds pixels 4l..4l+3 of the strip as two words, reads the 2k + 1 window rows ring by
// ring (LDS.64 + VIMNMX3.U16x2) and after each ring widens the running maximum by single-pixel steps: the neighbours' edge
// pixels arrive by two shuffles, PRMT lines the three shifted pairs up, VIMNMX3 takes the maximum.  Garbage creeps in from the
// strip's ends one pixel per step, k <= kZgHalo pixels in all, so the strip's own columns are exact.  Rows whose whole window is
// black (most of a colour-depth MIP) are skipped.
constexpr int kZgTH = 32;
constexpr int kZgStrip = 96;
constexpr int kZgHalo = 16;
constexpr int kZgWords = (kZgStrip + 2 * kZgHalo) / 2;      // 64 words = 128 pixels per staged row

__device__ __forceinline__ uint32_t vmax3_u16x2(uint32_t a, uint32_t b, uint32_t c) { return __vimax3_u16x2(a, b, c); }

template <bool OUT_RGB>
__global__ void __launch_bounds__(256) shape_target_derive_kernel(const uint8_t *__restrict__ target, int W, int H, RectSet rects, int threshold,
                                                                  DiscRings rings, const uint16_t *__restrict__ slice_tab,
                                                                  uint16_t *__restrict__ zslice, uint32_t *__restrict__ tsig, int bpitch,
                                                                  uint8_t *__restrict__ rgb_out)
{
    extern __shared__ uint32_t s_in[];                         // [3][rows][kZgWords]
    __shared__ uint32_t s_sig[kZgTH][4];
    __shared__ int s_rowpre[kZgTH + 2 * kZgHalo + 2];          // prefix sums of "row has a non-black pixel"
    const int k = rings.k;
    const int rows = kZgTH + 2 * k;
    const int64_t img = blockIdx.z;
    const int x0 = blockIdx.x * kZgStrip, y0 = blockIdx.y * kZgTH;
    const int xin = x0 - kZgHalo, yin = y0 - k;
    const uint8_t *src = target + (size_t) img * W * H * 3;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    if (tid < kZgTH * 4) s_sig[0][tid] = 0;
    if (tid <= rows) s_rowpre[tid] = 0;
    __syncthreads();

    // ---- stage: one pixel pair per thread and step (only tiles that touch a label rectangle test their pixels against them)
    bool near_rects = false;
    for (int i = 0; i < rects.n; i++)
        near_rects |= rects.x0[i] < xin + 2 * kZgWords && rects.x1[i] > xin && rects.y0[i] < yin + rows && rects.y1[i] > yin;
    int any = 0;
    for (int i = tid; i < rows * kZgWords; i += 256) {
        const int row = i / kZgWords, j = i % kZgWords;
        const int y = yin + row, x = xin + 2 * j;
        uint32_t wr = 0, wg = 0, wb = 0;
        if (y >= 0 && y < H) {
            const uint8_t *p = src + ((size_t) y * W + x) * 3;
#pragma unroll
            for (int e = 0; e < 2; e++) {
                const int xx = x + e;
                if (xx < 0 || xx >= W) continue;
                const int r = p[3 * e], g = p[3 * e + 1], b = p[3 * e + 2];
                const bool keep = (r > threshold || g > threshold || b > threshold) && !(near_rects && shape_in_rects(rects, xx, y));
                if (!keep) continue;
                wr |= (uint32_t) r << (16 * e); wg |= (uint32_t) g << (16 * e); wb |= (uint32_t) b << (16 * e);
                const int sx = xx - x0, sy = y - y0;
                if (!OUT_RGB && sx >= 0 && sx < kZgStrip && sy >= 0 && sy < kZgTH) atomicOr(&s_sig[sy][sx >> 5], 1u << (sx & 31));
            }
        }
        s_in[(0 * rows + row) * kZgWords + j] = wr;
        s_in[(1 * rows + row) * kZgWords + j] = wg;
        s_in[(2 * rows + row) * kZgWords + j] = wb;
        if (wr | wg | wb) { any = 1; s_rowpre[row + 1] = 1; }       // benign race: every writer stores 1
    }
    any = __syncthreads_or(any);

    if (!OUT_RGB) {
        // the target's signal bitmap of this tile (row layout, 32 pixels per word; x0 is a multiple of 32)
        // (the last strip also clears the row's pad words)
        const int nw = blockIdx.x + 1 == gridDim.x ? bpitch - (x0 >> 5) : 3;
        for (int i = tid; i < kZgTH * nw; i += 256) {
            const int sy = i / nw, wi = i % nw;
            const int y = y0 + sy, wcol = (x0 >> 5) + wi;
            if (y < H && wcol < bpitch) tsig[((size_t) img * H + y) * bpitch + wcol] = wi < 3 ? s_sig[sy][wi] : 0u;
        }
    }
    if (!any) {
        // nothing above the threshold anywhere near: the tile's output is black
        for (int i = tid; i < kZgTH * kZgStrip; i += 256) {
            const int y = y0 + i / kZgStrip, x = x0 + i % kZgStrip;
            if (y >= H || x >= W) continue;
            if (OUT_RGB) { uint8_t *o = rgb_out + (((size_t) img * H + y) * W + x) * 3; o[0] = o[1] = o[2] = 0; }
            else zslice[((size_t) img * H + y) * W + x] = 0;
        }
        return;
    }
    if (tid == 0) {
        int acc = 0;
        for (int r = 0; r < rows; r++) { acc += s_rowpre[r + 1]; s_rowpre[r + 1] = acc; }
    }
    __syncthreads();

    for (int ro = warp; ro < kZgTH; ro += 8) {
        const int y = y0 + ro;
        if (y >= H) break;
        uint32_t res[3][2] = {{0u, 0u}, {0u, 0u}, {0u, 0u}};
        if (s_rowpre[ro + 2 * k + 1] - s_rowpre[ro] > 0) {
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const uint32_t *base = s_in + ((size_t) c * rows + ro + k) * kZgWords + 2 * lane;      // the window's centre row, this lane's words
                uint32_t X0 = 0, X1 = 0;
                int dy = 0;
                for (int i = 0; i < rings.n; i++) {
                    const int h = rings.h[i];
                    for (; dy <= h; dy++) {
                        const uint2 a = *reinterpret_cast<const uint2 *>(base - dy * kZgWords);
                        const uint2 b = *reinterpret_cast<const uint2 *>(base + dy * kZgWords);
                        X0 = vmax3_u16x2(X0, a.x, b.x);
                        X1 = vmax3_u16x2(X1, a.y, b.y);
                    }
                    for (int s = rings.d[i]; s > 0; s--) {
                        uint32_t left = __shfl_up_sync(0xffffffffu, X1, 1), right = __shfl_down_sync(0xffffffffu, X0, 1);
                        if (lane == 0) left = 0;
                        if (lane == 31) right = 0;
                        const uint32_t A0 = __byte_perm(left, X0, 0x5432);      // pixels (4l - 1, 4l)
                        const uint32_t B0 = __byte_perm(X0, X1, 0x5432);        // pixels (4l + 1, 4l + 2)
                        const uint32_t B1 = __byte_perm(X1, right, 0x5432);     // pixels (4l + 3, 4l + 4)
                        X0 = vmax3_u16x2(A0, X0, B0);
                        X1 = vmax3_u16x2(B0, X1, B1);
                    }
                }
                res[c][0] = X0; res[c][1] = X1;
            }
        }
        // this lane's four pixels: strip columns 4l - kZgHalo .. + 3
        const int sx = 4 * lane - kZgHalo;
        if (sx < 0 || sx >= kZgStrip) continue;
        const int x = x0 + sx;
        if (OUT_RGB) {
#pragma unroll
            for (int e = 0; e < 4; e++) {
                if (x + e >= W) break;
                uint8_t *o = rgb_out + (((size_t) img * H + y) * W + x + e) * 3;
                o[0] = (uint8_t) ((res[0][e >> 1] >> (16 * (e & 1))) & 0xFFFFu);
                o[1] = (uint8_t) ((res[1][e >> 1] >> (16 * (e & 1))) & 0xFFFFu);
                o[2] = (uint8_t) ((res[2][e >> 1] >> (16 * (e & 1))) & 0xFFFFu);
            }
        } else {
            uint32_t sl[4];
#pragma unroll
            for (int e = 0; e < 4; e++) {
                const int r = (int) ((res[0][e >> 1] >> (16 * (e & 1))) & 0xFFFFu);
                const int g = (int) ((res[1][e >> 1] >> (16 * (e & 1))) & 0xFFFFu);
                const int b = (int) ((res[2][e >> 1] >> (16 * (e & 1))) & 0xFFFFu);
                sl[e] = (r > threshold || g > threshold || b > threshold) ? (uint32_t) slice_of(slice_tab, r, g, b) : 0u;   // mask(threshold) then slice
            }
            uint16_t *o = zslice + ((size_t) img * H + y) * W + x;
            if ((W & 1) == 0 && x + 3 < W) {
                *reinterpret_cast<uint32_t *>(o) = sl[0] | (sl[1] << 16);
                *reinterpret_cast<uint32_t *>(o + 2) = sl[2] | (sl[3] << 16);
            } else {
#pragma unroll
                for (int e = 0; e < 4; e++) if (x + e < W) o[e] = (uint16_t) sl[e];
            }
        }
    }
}

// target side of a pair when the caller supplies the zgap image: zslice = slice number of mask(threshold)(zgap), tsig as above
__global__ void __launch_bounds__(256) target_planes_kernel(const uint8_t *__restrict__ target, const uint8_t *__restrict__ zgap, int W, int H,
                                                            RectSet rects, int threshold, int bpitch, const uint16_t *__restrict__ slice_tab,
                                                            uint16_t *__restrict__ zslice, uint32_t *__restrict__ tsig)
{
    const int y = blockIdx.x;
    const int64_t img = blockIdx.y;
    const uint8_t *trow = target + ((size_t) img * H + y) * W * 3;
    const uint8_t *zrow = zgap + ((size_t) img * H + y) * W * 3;
    uint16_t *zs = zslice + ((size_t) img * H + y) * W;
    uint32_t *ts = tsig + ((size_t) img * H + y) * bpitch;
    const int lane = threadIdx.x & 31;
    for (int x0 = (threadIdx.x >> 5) * 32; x0 < bpitch * 32; x0 += (int) blockDim.x) {
        const int x = x0 + lane;
        bool sig = false;
        if (x < W) {
            const int r = trow[3 * x], g = trow[3 * x + 1], b = trow[3 * x + 2];
            sig = !shape_in_rects(rects, x, y) && (r > threshold || g > threshold || b > threshold);
            const int zr = zrow[3 * x], zg = zrow[3 * x + 1], zb = zrow[3 * x + 2];
            int sl = 0;
            if (zr > threshold || zg > threshold || zb > threshold) sl = slice_of(slice_tab, zr, zg, zb);   // mask(threshold) then slice
            zs[x] = (uint16_t) sl;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, sig);
        if (lane == 0) ts[x0 >> 5] = bal;
    }
}

// ------------------------------------------------------------------------------------------------------------------ mask side
// createShapeMatchCDSAlgorithmProvider :96-111 needs of the two dilations of Q (the label-cleared query) only
//     max20(Q) == black            <=>  no non-black pixel of Q inside the r = 20 disc                              = !dil20(N)
//     gray(max60(Q)) > 0           <=>  the three channel maxima over the r = 60 disc add up to >= 2 (gray_of above)
//                                  <=>  dil60(B2) | at least two of dil60(A_r), dil60(A_g), dil60(A_b)
// with the bitmaps N = "some channel > 0", B2 = "some channel >= 2", A_c = "channel c >= 1" -- binary dilations, 64 pixels per
// lane.  Scratch bitmaps are [which][mask][H][bpitch] with which = 0 (N, r = 20) and 1..4 (B2, A_r, A_g, A_b, r = 60).
constexpr int kMaskBitmaps = 5;

// per (mask, row): the five bitmaps, QM = gray(Q) > 2 count (counters[m][0]), gap-list length (counters[m][2]), row flags
__global__ void __launch_bounds__(256) shape_mask_bits_kernel(const uint8_t *__restrict__ rgb, int n_masks, int W, int H, int bpitch, RectSet rects,
                                                              const uint32_t *__restrict__ roi_bits, uint32_t *__restrict__ bits,
                                                              uint8_t *__restrict__ rowany, unsigned long long *__restrict__ counters)
{
    const int y = blockIdx.x, m = blockIdx.y;
    const uint8_t *row = rgb + ((size_t) m * H + y) * W * 3;
    const size_t plane = (size_t) n_masks * H * bpitch;
    uint32_t *out = bits + ((size_t) m * H + y) * bpitch;
    const int lane = threadIdx.x & 31;
    int qm_cnt = 0, list_cnt = 0, nz = 0;
    for (int x0 = (threadIdx.x >> 5) * 32; x0 < bpitch * 32; x0 += (int) blockDim.x) {
        const int x = x0 + lane;
        bool n = false, b2 = false, ar = false, ag = false, ab = false;
        if (x < W && !shape_in_rects(rects, x, y)) {
            const int r = row[3 * x], g = row[3 * x + 1], b = row[3 * x + 2];
            n = (r | g | b) != 0; b2 = r >= 2 || g >= 2 || b >= 2; ar = r >= 1; ag = g >= 1; ab = b >= 1;
            if (n) {
                qm_cnt += gray_of(r, g, b) > 2 ? 1 : 0;
                const int xs = W - 1 - x;
                const bool keep = !roi_bits || ((roi_bits[(size_t) y * bpitch + (x >> 5)] >> (x & 31)) & 1u);
                const bool keep_m = !roi_bits || ((roi_bits[(size_t) y * bpitch + (xs >> 5)] >> (xs & 31)) & 1u);
                list_cnt += (keep || keep_m) ? 1 : 0;
            }
        }
        const unsigned wn = __ballot_sync(0xffffffffu, n), w2 = __ballot_sync(0xffffffffu, b2);
        const unsigned wr = __ballot_sync(0xffffffffu, ar), wg = __ballot_sync(0xffffffffu, ag), wb = __ballot_sync(0xffffffffu, ab);
        if (lane == 0) {
            const int j = x0 >> 5;
            out[j] = wn; out[plane + j] = w2; out[2 * plane + j] = wr; out[3 * plane + j] = wg; out[4 * plane + j] = wb;
        }
        nz |= wn != 0;
    }
    qm_cnt = __reduce_add_sync(0xffffffffu, qm_cnt);
    list_cnt = __reduce_add_sync(0xffffffffu, list_cnt);
    if (lane == 0) {
        if (qm_cnt) atomicAdd(&counters[4 * m + 0], (unsigned long long) qm_cnt);
        if (list_cnt) atomicAdd(&counters[4 * m + 2], (unsigned long long) list_cnt);
    }
    const int any = __syncthreads_or(nz);
    if (threadIdx.x == 0) rowany[(size_t) m * H + y] = (uint8_t) (any != 0);
}

// binary disc dilation of bitmap `which` of every mask: one warp per output row, lane j = pixels 64j..64j+63 (two words).
__global__ void __launch_bounds__(256) shape_mask_dilate_kernel(const uint32_t *__restrict__ bits, const uint8_t *__restrict__ rowany, int n_masks, int H,
                                                                int bpitch, DiscRings rings20, DiscRings rings60, uint32_t *__restrict__ dil)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int y = blockIdx.x * 8 + warp;
    const int which = blockIdx.y % kMaskBitmaps, m = blockIdx.y / kMaskBitmaps;
    if (y >= H) return;
    const DiscRings &rings = which == 0 ? rings20 : rings60;
    const int k = rings.k;
    const size_t plane = (size_t) n_masks * H * bpitch;
    const uint32_t *in = bits + which * plane + (size_t) m * H * bpitch;
    uint32_t *out = dil + which * plane + ((size_t) m * H + y) * bpitch;
    const int np = bpitch / 2;
    // rows of the window that hold anything at all
    bool some = false;
    for (int r = y - k + lane; r <= y + k; r += 32)
        if (r >= 0 && r < H && rowany[(size_t) m * H + r]) some = true;
    if (!__any_sync(0xffffffffu, some)) {
        if (lane < np) *reinterpret_cast<uint2 *>(out + 2 * lane) = make_uint2(0u, 0u);
        return;
    }
    uint32_t lo = 0, hi = 0;
    int dy = 0;
    for (int i = 0; i < rings.n; i++) {
        const int h = rings.h[i];
        for (; dy <= h; dy++) {
            if (lane < np) {
                if (y - dy >= 0) { const uint2 a = __ldg(reinterpret_cast<const uint2 *>(in + (size_t) (y - dy) * bpitch) + lane); lo |= a.x; hi |= a.y; }
                if (dy > 0 && y + dy < H) { const uint2 b = __ldg(reinterpret_cast<const uint2 *>(in + (size_t) (y + dy) * bpitch) + lane); lo |= b.x; hi |= b.y; }
            }
        }
        for (int s = rings.d[i]; s > 0; s--) {
            uint32_t lefthi = __shfl_up_sync(0xffffffffu, hi, 1), rightlo = __shfl_down_sync(0xffffffffu, lo, 1);
            if (lane == 0) lefthi = 0;
            if (lane == 31) rightlo = 0;
            const uint32_t nlo = lo | __funnelshift_l(lefthi, lo, 1) | __funnelshift_r(lo, hi, 1);
            const uint32_t nhi = hi | __funnelshift_l(lo, hi, 1) | __funnelshift_r(hi, rightlo, 1);
            lo = nlo; hi = nhi;
        }
    }
    if (lane < np) *reinterpret_cast<uint2 *>(out + 2 * lane) = make_uint2(lo, hi);
}

// HE = !dil20(N) & (dil60(B2) | majority(dil60(A_r), dil60(A_g), dil60(A_b))) inside the image; he_n = HE & ROI,
// he_m = mirror(HE) & ROI (the ROI is not mirrored with the query, Shape2DMatch...:205-218); counters[m][1] += |HE|.
__global__ void __launch_bounds__(64) shape_mask_finish_kernel(const uint32_t *__restrict__ dil, int n_masks, int W, int H, int bpitch,
                                                               const uint32_t *__restrict__ roi_bits, uint32_t *const *__restrict__ he_n_ptrs,
                                                               uint32_t *const *__restrict__ he_m_ptrs, unsigned long long *__restrict__ counters)
{
    __shared__ uint32_t s_he[66];
    const int y = blockIdx.x, m = blockIdx.y, j = threadIdx.x;
    const size_t plane = (size_t) n_masks * H * bpitch;
    const uint32_t *d = dil + ((size_t) m * H + y) * bpitch;
    uint32_t he = 0;
    if (j < bpitch) {
        const uint32_t dn = d[j], d2 = d[plane + j], dr = d[2 * plane + j], dg = d[3 * plane + j], db = d[4 * plane + j];
        he = ~dn & (d2 | (dr & dg) | (dr & db) | (dg & db));
        const int rem = W - 32 * j;                                           // pixels of this word that are inside the image
        if (rem <= 0) he = 0;
        else if (rem < 32) he &= (1u << rem) - 1u;
    }
    s_he[j + 1] = he;
    if (j == 0) { s_he[0] = 0; s_he[65] = 0; }
    int cnt = __popc(he);
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((j & 31) == 0 && cnt) atomicAdd(&counters[4 * m + 1], (unsigned long long) cnt);
    __syncthreads();
    if (j >= bpitch) return;
    const uint32_t roi = roi_bits ? roi_bits[(size_t) y * bpitch + j] : 0xffffffffu;
    he_n_ptrs[m][(size_t) y * bpitch + j] = he & roi;
    // mirrored word j: output pixel x = 32 j + b takes HE(W - 1 - x); the 32 source pixels start at lo = W - 32 - 32 j
    const int lo = W - 32 - 32 * j;
    const int idx = lo >> 5, off = lo & 31;                                   // floor division: lo may be negative
    const uint32_t w0 = (idx >= 0 && idx < 64) ? s_he[idx + 1] : 0u, w1 = (idx + 1 >= 0 && idx + 1 < 64) ? s_he[idx + 2] : 0u;
    const uint32_t v = __funnelshift_r(w0, w1, off);
    he_m_ptrs[m][(size_t) y * bpitch + j] = __brev(v) & roi;
}

// gap list entry for every pixel with Q != black that the ROI keeps in at least one orientation:
//     x | y << 11 | (slice(Q) - 1) << 21 | QM << 29 | keep_normal << 30 | keep_mirrored << 31
__global__ void __launch_bounds__(256) shape_mask_list_kernel(const uint8_t *__restrict__ rgb, int W, int H, int bpitch, RectSet rects,
                                                              const uint32_t *__restrict__ roi_bits, const uint16_t *__restrict__ slice_tab,
                                                              uint32_t *const *__restrict__ list_ptrs, unsigned long long *__restrict__ counters)
{
    const int y = blockIdx.x, m = blockIdx.y;
    const uint8_t *row = rgb + ((size_t) m * H + y) * W * 3;
    uint32_t *list = list_ptrs[m];
    for (int x = threadIdx.x; x < W; x += blockDim.x) {
        if (shape_in_rects(rects, x, y)) continue;
        const int r = row[3 * x], g = row[3 * x + 1], b = row[3 * x + 2];
        if ((r | g | b) == 0) continue;
        const int xs = W - 1 - x;
        const bool keep = !roi_bits || ((roi_bits[(size_t) y * bpitch + (x >> 5)] >> (x & 31)) & 1u);
        const bool keep_m = !roi_bits || ((roi_bits[(size_t) y * bpitch + (xs >> 5)] >> (xs & 31)) & 1u);
        if (!keep && !keep_m) continue;
        const uint32_t qm = gray_of(r, g, b) > 2 ? 1u : 0u;
        const uint32_t e = (uint32_t) x | ((uint32_t) y << 11) | ((uint32_t) (slice_of(slice_tab, r, g, b) - 1) << 21) | (qm << 29) |
                           ((uint32_t) keep << 30) | ((uint32_t) keep_m << 31);
        const unsigned long long slot = atomicAdd(&counters[4 * m + 3], 1ull);
        list[slot] = e;
    }
}

// the label-cleared ROI as a bitmap: bit set where the ROI pixel is not black (ColorTransformation.mask(pt, p, m) :134-143)
__global__ void __launch_bounds__(256) shape_roi_bits_kernel(const uint8_t *__restrict__ roi, int W, int H, int bpitch, RectSet rects, uint32_t *__restrict__ bits)
{
    const int y = blockIdx.x;
    const int lane = threadIdx.x & 31;
    for (int x0 = (threadIdx.x >> 5) * 32; x0 < bpitch * 32; x0 += (int) blockDim.x) {
        const int x = x0 + lane;
        bool keep = false;
        if (x < W && !shape_in_rects(rects, x, y)) keep = (roi[((size_t) y * W + x) * 3] | roi[((size_t) y * W + x) * 3 + 1] | roi[((size_t) y * W + x) * 3 + 2]) != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) bits[(size_t) y * bpitch + (x0 >> 5)] = bal;
    }
}

// ------------------------------------------------------------------------------------------------------------------ pair kernel
// pair_slot = index of the pair's target inside the window's planes
__global__ void __launch_bounds__(256) shape_pair_kernel(const ShapeMaskDesc *__restrict__ masks, const int32_t *__restrict__ pair_mask,
                                                         const int32_t *__restrict__ pair_slot,
                                                         const uint16_t *__restrict__ zslice, const uint16_t *__restrict__ grad,
                                                         const uint32_t *__restrict__ tsig, int W, int H, int bpitch, int mirror,
                                                         long long *__restrict__ gap_out, long long *__restrict__ he_out, uint8_t *__restrict__ mir_out)
{
    __shared__ long long s_red[4][8];
    const int64_t pr = blockIdx.x;
    const int64_t t = pair_slot[pr];
    const ShapeMaskDesc md = masks[pair_mask[pr]];
    const uint16_t *zs = zslice + (size_t) t * W * H;
    const uint16_t *gr = grad + (size_t) t * W * H;
    const uint32_t *ts = tsig + (size_t) t * H * bpitch;
    long long gap_n = 0, gap_m = 0, he_n = 0, he_m = 0;
    for (int i = threadIdx.x; i < md.n_gap; i += blockDim.x) shape_gap_entry(__ldg(md.gap_list + i), zs, gr, W, mirror, gap_n, gap_m);
    const int n_words = H * bpitch;
    for (int i = threadIdx.x; i < n_words; i += blockDim.x) shape_he_word(md, ts, i, mirror, he_n, he_m);
    long long v[4] = {gap_n, gap_m, he_n, he_m};
#pragma unroll
    for (int k = 0; k < 4; k++) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], off);
        if ((threadIdx.x & 31) == 0) s_red[k][threadIdx.x >> 5] = v[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        long long tot[4] = {0, 0, 0, 0};
        for (int k = 0; k < 4; k++) for (int w = 0; w < 8; w++) tot[k] += s_red[k][w];
        long long g, h;
        const int mir = shape_pick(tot, mirror, g, h);
        gap_out[pr] = g; he_out[pr] = h; mir_out[pr] = (uint8_t) mir;
    }
}

// per-device constants of the shape path: the colour LUT in constant memory and the slice table
static cds_status ensure_shape_tables(cds_ctx *ctx, DevState &ds)
{
    if (ds.d_slice_tab) return CDS_OK;
    cds_status st = ctx->check(cudaSetDevice(ds.dev), "cudaSetDevice");
    if (st == CDS_OK) st = ctx->check(cudaMemcpyToSymbol(c_shape_lut, kColorDepthLut, sizeof(kColorDepthLut)), "lut upload");
    uint16_t *tab = nullptr;
    if (st == CDS_OK) st = ctx->check(cudaMalloc(&tab, kSliceTabEntries * sizeof(uint16_t)), "cudaMalloc(slice table)");
    if (st == CDS_OK) {
        build_slice_table_kernel<<<(kSliceTabEntries + 255) / 256, 256, 0, ds.stream>>>(tab);
        st = ctx->check(cudaGetLastError(), "build_slice_table_kernel");
    }
    if (st == CDS_OK) st = ctx->check(cudaStreamSynchronize(ds.stream), "slice table");
    if (st != CDS_OK) { if (tab) cudaFree(tab); return st; }
    ds.d_slice_tab = tab;
    return CDS_OK;
}

void shape_release_dev(DevState &ds)
{
    if (ds.d_slice_tab) cudaFree(ds.d_slice_tab);
    ds.d_slice_tab = nullptr;
    for (cudaEvent_t e : ds.shape_timing) cudaEventDestroy(e);
    ds.shape_timing.clear();
    if (ds.h_pinned2) cudaFreeHost(ds.h_pinned2);
    ds.h_pinned2 = nullptr;
    ds.h_pinned2_bytes = 0;
}

// launches the fused derive kernel for n images; false when the disc is outside its envelope
template <bool OUT_RGB>
static bool launch_target_derive(const uint8_t *target, int64_t n, int W, int H, const RectSet &rects, int threshold, const DiscSpec &disc,
                                 const uint16_t *slice_tab, uint16_t *zslice, uint32_t *tsig, int bpitch, uint8_t *rgb_out, cudaStream_t s)
{
    if (disc.k > kZgHalo || disc.k < 0) return false;
    const DiscRings rings = make_rings(disc);
    const size_t smem = (size_t) 3 * (kZgTH + 2 * disc.k) * kZgWords * sizeof(uint32_t);
    auto kern = shape_target_derive_kernel<OUT_RGB>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    for (int64_t i0 = 0; i0 < n; i0 += 32768) {
        const int64_t cnt = std::min<int64_t>(32768, n - i0);
        dim3 grid((W + kZgStrip - 1) / kZgStrip, (H + kZgTH - 1) / kZgTH, (unsigned) cnt);
        kern<<<grid, 256, smem, s>>>(target + (size_t) i0 * W * H * 3, W, H, rects, threshold, rings, slice_tab,
                                     zslice ? zslice + (size_t) i0 * W * H : nullptr, tsig ? tsig + (size_t) i0 * H * bpitch : nullptr, bpitch,
                                     rgb_out ? rgb_out + (size_t) i0 * W * H * 3 : nullptr);
    }
    return true;
}

}  // namespace cds

// ------------------------------------------------------------------------------------------------------------------ C ABI
#define SH_TRY(expr) do { cds_status _s = (expr); if (_s != CDS_OK) return _s; } while (0)
#define SH_CUDA(ctx, expr) SH_TRY((ctx)->check((expr), #expr))

void cds::launch_shape_target_planes(const cds_shape_maskset *sms, const DevState &ds, const uint8_t *target, const uint8_t *zgap, int64_t n,
                                     uint16_t *zslice, uint32_t *tsig, cudaStream_t s)
{
    if (zgap) {
        target_planes_kernel<<<dim3(sms->H, (unsigned) n), 256, 0, s>>>(target, zgap, sms->W, sms->H, sms->rects, sms->query_threshold, sms->bpitch,
                                                                       ds.d_slice_tab, zslice, tsig);
    } else {
        // the zgap image the reference's tests derive: maxFilter(10)(mask(threshold)(clearLabels(target))), never materialised
        launch_target_derive<false>(target, n, sms->W, sms->H, sms->rects, sms->query_threshold, make_disc(10), ds.d_slice_tab, zslice, tsig,
                                    sms->bpitch, nullptr, s);
    }
}

static RectSet to_rectset(const cds_rect *rects, int n)
{
    RectSet r{};
    r.n = n;
    for (int i = 0; i < n; i++) { r.x0[i] = rects[i].x0; r.y0[i] = rects[i].y0; r.x1[i] = rects[i].x1; r.y1[i] = rects[i].y1; }
    return r;
}

namespace {
// frees pooled blocks on scope exit, after the device's streams have drained
struct PoolGuard {
    DevState *ds;
    std::vector<void *> ptrs;
    explicit PoolGuard(DevState *d) : ds(d) {}
    cudaError_t alloc(void **p, size_t bytes) { cudaError_t e = ds->pool.alloc(p, bytes); if (e == cudaSuccess) ptrs.push_back(*p); return e; }
    ~PoolGuard()
    {
        if (ptrs.empty()) return;
        cudaSetDevice(ds->dev);
        cudaStreamSynchronize(ds->copy_stream);
        cudaStreamSynchronize(ds->stream);
        for (void *p : ptrs) ds->pool.free(p);
    }
};
}  // namespace

extern "C" cds_status cds_shape_maskset_create(cds_ctx *ctx, int32_t width, int32_t height, int32_t query_threshold, int32_t border,
                                               int32_t mirror, const cds_rect *rects, int32_t n_rects, const uint8_t *roi_rgb,
                                               cds_shape_maskset **out)
{
    return cds::abi_guard("cds_shape_maskset_create", [&]() -> cds_status {
        if (!ctx || !out) { set_tls_error("cds_shape_maskset_create: NULL argument"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        *out = nullptr;
        if (width <= 0 || height <= 0 || n_rects < 0 || n_rects > CDS_MAX_RECTS || (n_rects > 0 && !rects))
            return ctx->fail(CDS_ERR_BAD_ARG, "cds_shape_maskset_create: bad arguments");
        if (width > 2048 || height > 1024) return ctx->fail(CDS_ERR_UNSUPPORTED, "cds_shape_maskset_create: images larger than 2048 x 1024 are not supported");
        if (border != 0) return ctx->fail(CDS_ERR_UNSUPPORTED, "cds_shape_maskset_create: only border = 0 is supported");
        auto sms = new cds_shape_maskset();
        sms->ctx = ctx; sms->W = width; sms->H = height; sms->bpitch = occupancy_valid_pitch(width);   // row-layout bitmaps: one bit per pixel, 32-pixel words
        sms->query_threshold = query_threshold; sms->mirror = mirror ? 1 : 0;
        sms->rects = to_rectset(rects, n_rects);
        sms->dev.resize(ctx->devs.size());
        DevState &d0 = ctx->devs[0];
        cds_status st = CDS_OK;
        for (DevState &ds : ctx->devs) if (st == CDS_OK) st = ensure_shape_tables(ctx, ds);
        if (st == CDS_OK) st = ctx->check(cudaSetDevice(d0.dev), "cudaSetDevice");
        if (st == CDS_OK && roi_rgb) {
            const size_t bytes = (size_t) width * height * 3;
            uint8_t *tmp = nullptr;
            st = ctx->check(cudaMalloc(&sms->d_roi_bits, (size_t) height * sms->bpitch * sizeof(uint32_t)), "cudaMalloc(roi)");
            if (st == CDS_OK) st = ctx->check(cudaMalloc(&tmp, bytes), "cudaMalloc(roi tmp)");
            if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(tmp, roi_rgb, bytes, cudaMemcpyHostToDevice, d0.stream), "roi H2D");
            if (st == CDS_OK) {
                shape_roi_bits_kernel<<<height, 256, 0, d0.stream>>>(tmp, width, height, sms->bpitch, sms->rects, sms->d_roi_bits);   // the ROI is label-cleared too (:97-101)
                st = ctx->check(cudaGetLastError(), "shape_roi_bits_kernel");
            }
            if (st == CDS_OK) st = ctx->check(cudaStreamSynchronize(d0.stream), "roi");
            if (tmp) cudaFree(tmp);
        }
        if (st != CDS_OK) { cds_shape_maskset_destroy(sms); return st; }
        *out = sms;
        return CDS_OK;
    });
}

extern "C" void cds_shape_maskset_destroy(cds_shape_maskset *sms)
{
    if (!sms) return;
    cds_ctx *ctx = sms->ctx;
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    for (size_t d = 0; d < sms->dev.size(); d++) {
        DevState &ds = ctx->devs[d];
        cudaSetDevice(ds.dev);
        cudaStreamSynchronize(ds.copy_stream);
        cudaStreamSynchronize(ds.stream);
        for (void *p : sms->dev[d].blocks) ds.pool.free(p);
        if (sms->dev[d].d_descs) cudaFree(sms->dev[d].d_descs);
    }
    if (sms->d_roi_bits) { cudaSetDevice(ctx->devs[0].dev); cudaFree(sms->d_roi_bits); }
    cudaGetLastError();
    delete sms;
}

extern "C" int32_t cds_shape_maskset_size(const cds_shape_maskset *sms) { return sms ? sms->n_masks : 0; }

// Masks are prepared on device 0 in batches: upload, bitmaps + counts (one read-back: the gap lists' lengths size the batch's block),
// the five binary dilations, HE bitmaps, gap lists; the finished block is then copied to the other devices.
extern "C" cds_status cds_shape_maskset_add_rgb(cds_shape_maskset *sms, const uint8_t *rgb, int32_t n, int64_t *qm_size_out, int64_t *he_size_out)
{
    return cds::abi_guard("cds_shape_maskset_add_rgb", [&]() -> cds_status {
        if (!sms) { set_tls_error("cds_shape_maskset_add_rgb: NULL mask set"); return CDS_ERR_BAD_ARG; }
        cds_ctx *ctx = sms->ctx;
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (n < 0 || (n > 0 && !rgb)) return ctx->fail(CDS_ERR_BAD_ARG, "cds_shape_maskset_add_rgb: bad arguments");
        if (n == 0) return CDS_OK;
        const int D = (int) ctx->devs.size();
        DevState &d0 = ctx->devs[0];
        SH_CUDA(ctx, cudaSetDevice(d0.dev));
        const int W = sms->W, H = sms->H, bpitch = sms->bpitch;
        const size_t px = (size_t) W * H, bytes = px * 3;
        const size_t bm_words = (size_t) H * bpitch;
        const int batch = std::min<int>(n, 64);
        const DiscRings rings20 = make_rings(make_disc(20)), rings60 = make_rings(make_disc(60));

        PoolGuard g0(&d0);
        uint8_t *d_raw = nullptr, *d_rowany = nullptr;
        uint32_t *d_bits = nullptr, *d_dil = nullptr;
        unsigned long long *d_cnt = nullptr;
        uint32_t **d_ptrs = nullptr;                        // [3][batch]: list, he_n, he_m pointers of the batch's masks
        SH_CUDA(ctx, g0.alloc((void **) &d_raw, (size_t) batch * bytes));
        SH_CUDA(ctx, g0.alloc((void **) &d_bits, (size_t) kMaskBitmaps * batch * bm_words * sizeof(uint32_t)));
        SH_CUDA(ctx, g0.alloc((void **) &d_dil, (size_t) kMaskBitmaps * batch * bm_words * sizeof(uint32_t)));
        SH_CUDA(ctx, g0.alloc((void **) &d_rowany, (size_t) batch * H));
        SH_CUDA(ctx, g0.alloc((void **) &d_cnt, (size_t) batch * 4 * sizeof(unsigned long long)));
        SH_CUDA(ctx, g0.alloc((void **) &d_ptrs, (size_t) 3 * batch * sizeof(uint32_t *)));
        std::vector<unsigned long long> cnt((size_t) batch * 4);
        std::vector<uint32_t *> h_ptrs((size_t) 3 * batch);

        for (int i0 = 0; i0 < n; i0 += batch) {
            const int nb = std::min(batch, n - i0);
            SH_CUDA(ctx, cudaSetDevice(d0.dev));
            SH_CUDA(ctx, cudaMemcpyAsync(d_raw, rgb + (size_t) i0 * bytes, (size_t) nb * bytes, cudaMemcpyHostToDevice, d0.stream));
            SH_CUDA(ctx, cudaMemsetAsync(d_cnt, 0, (size_t) nb * 4 * sizeof(unsigned long long), d0.stream));
            shape_mask_bits_kernel<<<dim3(H, nb), 256, 0, d0.stream>>>(d_raw, nb, W, H, bpitch, sms->rects, sms->d_roi_bits, d_bits, d_rowany, d_cnt);
            SH_CUDA(ctx, cudaGetLastError());
            SH_CUDA(ctx, cudaMemcpyAsync(cnt.data(), d_cnt, (size_t) nb * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, d0.stream));
            shape_mask_dilate_kernel<<<dim3((H + 7) / 8, nb * kMaskBitmaps), 256, 0, d0.stream>>>(d_bits, d_rowany, nb, H, bpitch, rings20, rings60, d_dil);
            SH_CUDA(ctx, cudaGetLastError());
            SH_CUDA(ctx, cudaStreamSynchronize(d0.stream));         // the list lengths (the dilation above is already running)
            // one block per batch and device: [he_n | he_m] per mask, then the gap lists
            size_t list_words = 0;
            for (int i = 0; i < nb; i++) list_words += (size_t) ((cnt[4 * i + 2] + 3) / 4 * 4);
            const size_t block_words = (size_t) nb * 2 * bm_words + std::max<size_t>(list_words, 4);
            std::vector<uint32_t *> block(D, nullptr);
            for (int d = 0; d < D; d++) {
                SH_CUDA(ctx, cudaSetDevice(ctx->devs[d].dev));
                void *p = nullptr;
                SH_CUDA(ctx, ctx->devs[d].pool.alloc(&p, block_words * sizeof(uint32_t)));
                sms->dev[d].blocks.push_back(p);
                block[d] = (uint32_t *) p;
            }
            SH_CUDA(ctx, cudaSetDevice(d0.dev));
            size_t lo = (size_t) nb * 2 * bm_words;
            std::vector<size_t> list_off(nb);
            for (int i = 0; i < nb; i++) {
                list_off[i] = lo;
                h_ptrs[i] = block[0] + lo;
                h_ptrs[batch + i] = block[0] + (size_t) i * 2 * bm_words;
                h_ptrs[2 * batch + i] = block[0] + (size_t) i * 2 * bm_words + bm_words;
                lo += (size_t) ((cnt[4 * i + 2] + 3) / 4 * 4);
            }
            SH_CUDA(ctx, cudaMemcpyAsync(d_ptrs, h_ptrs.data(), (size_t) 3 * batch * sizeof(uint32_t *), cudaMemcpyHostToDevice, d0.stream));
            shape_mask_finish_kernel<<<dim3(H, nb), 64, 0, d0.stream>>>(d_dil, nb, W, H, bpitch, sms->d_roi_bits, d_ptrs + batch, d_ptrs + 2 * batch, d_cnt);
            shape_mask_list_kernel<<<dim3(H, nb), 256, 0, d0.stream>>>(d_raw, W, H, bpitch, sms->rects, sms->d_roi_bits, d0.d_slice_tab, d_ptrs, d_cnt);
            SH_CUDA(ctx, cudaGetLastError());
            ctx->stats.kernel_launches += 4;
            SH_CUDA(ctx, cudaMemcpyAsync(cnt.data(), d_cnt, (size_t) nb * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, d0.stream));
            for (int d = 1; d < D; d++)
                SH_CUDA(ctx, cudaMemcpyPeerAsync(block[d], ctx->devs[d].dev, block[0], d0.dev, block_words * sizeof(uint32_t), d0.stream));
            SH_CUDA(ctx, cudaStreamSynchronize(d0.stream));
            for (int i = 0; i < nb; i++) {
                if (qm_size_out) qm_size_out[i0 + i] = (int64_t) cnt[4 * i + 0];
                if (he_size_out) he_size_out[i0 + i] = (int64_t) cnt[4 * i + 1];
                for (int d = 0; d < D; d++) {
                    ShapeMaskDesc md;
                    md.gap_list = block[d] + list_off[i];
                    md.he_n = block[d] + (size_t) i * 2 * bm_words;
                    md.he_m = md.he_n + bm_words;
                    md.n_gap = (int) cnt[4 * i + 2];
                    md.pad = 0;
                    sms->dev[d].h_descs.push_back(md);
                    sms->dev[d].dirty = true;
                }
            }
            sms->n_masks += nb;
        }
        return CDS_OK;
    });
}

extern "C" cds_status cds_make_zgap(cds_ctx *ctx, const uint8_t *rgb, int64_t n, int32_t width, int32_t height, int32_t threshold,
                                    double radius, const cds_rect *rects, int32_t n_rects, uint8_t *zgap_out)
{
    return cds::abi_guard("cds_make_zgap", [&]() -> cds_status {
        if (!ctx) { set_tls_error("cds_make_zgap: NULL ctx"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (n < 0 || (n > 0 && (!rgb || !zgap_out)) || width <= 0 || height <= 0 || n_rects < 0 || n_rects > CDS_MAX_RECTS || (n_rects > 0 && !rects))
            return ctx->fail(CDS_ERR_BAD_ARG, "cds_make_zgap: bad arguments");
        const DiscSpec disc = make_disc(radius);
        if (disc.k > 60) return ctx->fail(CDS_ERR_UNSUPPORTED, "cds_make_zgap: radius > 60 is not supported");
        DevState &d0 = ctx->devs[0];
        SH_CUDA(ctx, cudaSetDevice(d0.dev));
        const RectSet rs = to_rectset(rects, n_rects);
        const size_t bytes = (size_t) width * height * 3;
        const int64_t chunk = 32;
        PoolGuard g0(&d0);
        uint8_t *d_a = nullptr, *d_b = nullptr;
        SH_CUDA(ctx, g0.alloc((void **) &d_a, chunk * bytes));
        SH_CUDA(ctx, g0.alloc((void **) &d_b, chunk * bytes));
        for (int64_t i0 = 0; i0 < n; i0 += chunk) {
            const int64_t cnt = std::min<int64_t>(chunk, n - i0);
            SH_CUDA(ctx, cudaMemcpyAsync(d_a, rgb + (size_t) i0 * bytes, (size_t) cnt * bytes, cudaMemcpyHostToDevice, d0.stream));
            uint8_t *res = d_b;
            if (launch_target_derive<true>(d_a, cnt, width, height, rs, threshold, disc, nullptr, nullptr, nullptr, 0, d_b, d0.stream)) {
                ctx->stats.kernel_launches += 1;
            } else {
                clear_and_mask_kernel<<<148 * 4, 256, 0, d0.stream>>>(d_a, d_b, cnt, width, height, rs, threshold, 1);
                launch_max_filter(d_b, d_a, cnt, width, height, 3, disc, d0.stream);
                ctx->stats.kernel_launches += 2;
                res = d_a;
            }
            SH_CUDA(ctx, cudaGetLastError());
            SH_CUDA(ctx, cudaMemcpyAsync(zgap_out + (size_t) i0 * bytes, res, (size_t) cnt * bytes, cudaMemcpyDeviceToHost, d0.stream));
            SH_CUDA(ctx, cudaStreamSynchronize(d0.stream));
        }
        return CDS_OK;
    });
}

extern "C" cds_status cds_debug_slice_numbers(cds_ctx *ctx, const uint8_t *rgb, int64_t n, uint16_t *slices_out)
{
    return cds::abi_guard("cds_debug_slice_numbers", [&]() -> cds_status {
        if (!ctx) { set_tls_error("cds_debug_slice_numbers: NULL ctx"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (n < 0 || (n > 0 && (!rgb || !slices_out))) return ctx->fail(CDS_ERR_BAD_ARG, "cds_debug_slice_numbers: bad arguments");
        if (n == 0) return CDS_OK;
        DevState &d0 = ctx->devs[0];
        SH_TRY(ensure_shape_tables(ctx, d0));
        SH_CUDA(ctx, cudaSetDevice(d0.dev));
        PoolGuard g0(&d0);
        uint8_t *d_rgb = nullptr;
        uint16_t *d_out = nullptr;
        SH_CUDA(ctx, g0.alloc((void **) &d_rgb, (size_t) n * 3));
        SH_CUDA(ctx, g0.alloc((void **) &d_out, (size_t) n * sizeof(uint16_t)));
        SH_CUDA(ctx, cudaMemcpyAsync(d_rgb, rgb, (size_t) n * 3, cudaMemcpyHostToDevice, d0.stream));
        slice_numbers_kernel<<<148 * 8, 256, 0, d0.stream>>>(d_rgb, n, d0.d_slice_tab, d_out);
        SH_CUDA(ctx, cudaGetLastError());
        SH_CUDA(ctx, cudaMemcpyAsync(slices_out, d_out, (size_t) n * sizeof(uint16_t), cudaMemcpyDeviceToHost, d0.stream));
        SH_CUDA(ctx, cudaStreamSynchronize(d0.stream));
        return CDS_OK;
    });
}

namespace {

// Gradient PNG files inflated on the device, one warp per stream: a stream takes tens of milliseconds whatever else runs, so the rate is
// the number of streams in flight over that latency -- windows are as large as the call's size allows (2 048 targets: ~20 GB of
// window buffers per device; measured: profiles/r02_shape_files.txt)
constexpr int64_t kShapeWindowInflate = 2048;
constexpr int64_t kShapeWindowSmall = 32, kShapeWindowLarge = 128;      // targets per window: large calls use large windows (pair-kernel launches that fill the GPU)

// What one device holds while it works through its windows.
struct ShapeDevWork {
    uint8_t *d_t[2] = {nullptr, nullptr}, *d_z[2] = {nullptr, nullptr};
    uint16_t *d_grad[2] = {nullptr, nullptr};
    uint16_t *d_zslice = nullptr;
    uint32_t *d_tsig = nullptr;
    uint8_t *d_comp = nullptr;
    TiffStrip *d_strips = nullptr;
    uint8_t *d_pngraw = nullptr, *d_bps = nullptr;
    uint8_t *d_zstage = nullptr;            // device inflate: {jobs, bytes per sample, the files' zlib streams} of one window, as staged by the host
    int32_t *d_zstat = nullptr;             // ... per image: 0 or why the device refused the stream
    uint8_t *d_zfallback = nullptr;         // ... one image's scanlines inflated by the host after a refusal (+ its bytes per sample)
    int32_t *d_pm = nullptr, *d_ps = nullptr;
    long long *d_gap = nullptr, *d_he = nullptr;
    uint8_t *d_mir = nullptr;
    std::vector<int32_t> pm, ps;            // this device's pairs in window order
    std::vector<int64_t> where;             // their positions in the caller's arrays
    std::vector<long long> h_gap, h_he;
    std::vector<uint8_t> h_mir;
    int64_t windows = 0;
};

}  // namespace

// Targets either as pixels (target_rgb) or as TIFF files stored back to back (blob + offsets, decoded on the device).
static cds_status shape_score_pairs_impl(cds_ctx *ctx, const cds_shape_maskset *sms_c, const uint8_t *target_rgb,
                                         const uint8_t *blob, const int64_t *offsets, const uint16_t *gradient,
                                         const uint8_t *png_blob, const int64_t *png_offsets,
                                         const uint8_t *zgap_rgb, const uint8_t *has_variants, int64_t n_targets,
                                         const int32_t *pair_mask, const int64_t *pair_target, int64_t n_pairs,
                                         int64_t *gap_out, int64_t *high_expr_out, uint8_t *mirrored_out)
{
    if (!ctx || !sms_c) { set_tls_error("cds_shape_score_pairs: NULL argument"); return CDS_ERR_BAD_ARG; }
    std::lock_guard<std::recursive_mutex> lk(ctx->mu);
    cds_shape_maskset *sms = const_cast<cds_shape_maskset *>(sms_c);
    if (sms->ctx != ctx) return ctx->fail(CDS_ERR_BAD_ARG, "cds_shape_score_pairs: mask set belongs to another context");
    if (n_pairs < 0 || n_targets < 0) return ctx->fail(CDS_ERR_BAD_ARG, "cds_shape_score_pairs: negative count");
    if (n_pairs == 0) return CDS_OK;
    if (!pair_mask || !pair_target || !gap_out || !high_expr_out || !mirrored_out) return ctx->fail(CDS_ERR_BAD_ARG, "cds_shape_score_pairs: NULL pair arrays");
    const int M = sms->n_masks;
    // pairs per target (counting sort by target keeps the caller's order inside a target)
    std::vector<int64_t> tstart((size_t) n_targets + 1, 0);
    bool any_scored = false;
    for (int64_t i = 0; i < n_pairs; i++) {
        if (pair_mask[i] < 0 || pair_mask[i] >= M || pair_target[i] < 0 || pair_target[i] >= n_targets)
            return ctx->fail(CDS_ERR_BAD_ARG, "cds_shape_score_pairs: pair index out of range");
        if (!has_variants || has_variants[pair_target[i]]) { any_scored = true; tstart[pair_target[i] + 1]++; }
        else { gap_out[i] = -1; high_expr_out[i] = -1; mirrored_out[i] = 0; }      // missing gradient / zgap supplier: (-1, -1, not mirrored), Shape2DMatch...:155-158
    }
    // a missing gradient can only be expressed through has_variants; a NULL gradient array with scorable pairs is an error
    const bool from_files = blob != nullptr && offsets != nullptr;
    const bool from_png = png_blob != nullptr && png_offsets != nullptr;
    if (any_scored && ((!target_rgb && !from_files) || (!gradient && !from_png))) return ctx->fail(CDS_ERR_BAD_ARG, "cds_shape_score_pairs: target / gradient images are NULL");
    ctx->stats = cds_search_stats{};
    if (!any_scored) return CDS_OK;
    if (from_files)
        for (int64_t i = 0; i <= n_targets; i++)
            if (offsets[i] < 0 || (i > 0 && offsets[i] < offsets[i - 1])) return ctx->fail(CDS_ERR_BAD_ARG, "cds_shape_score_pairs_tiff: offsets must be non-decreasing");
    for (int64_t t = 0; t < n_targets; t++) tstart[t + 1] += tstart[t];
    const int64_t n_scored = tstart[n_targets];
    std::vector<int64_t> order((size_t) n_scored);
    {
        std::vector<int64_t> cur(tstart.begin(), tstart.end() - 1);
        for (int64_t i = 0; i < n_pairs; i++)
            if (!has_variants || has_variants[pair_target[i]]) order[cur[pair_target[i]]++] = i;
    }
    std::vector<int64_t> active;                    // targets that are scored at all, ascending
    for (int64_t t = 0; t < n_targets; t++) if (tstart[t + 1] > tstart[t]) active.push_back(t);

    const int W = sms->W, H = sms->H, bpitch = sms->bpitch;
    const size_t px = (size_t) W * H, bytes = px * 3;
    const size_t bm_words = (size_t) H * bpitch;
    const int D = (int) ctx->devs.size();
    const bool dev_inflate = png_blob != nullptr && png_offsets != nullptr && ctx->device_inflate != 0;
    int64_t win = (int64_t) active.size() >= 4 * kShapeWindowLarge * D ? kShapeWindowLarge : kShapeWindowSmall;
    if (dev_inflate) {
        // the largest of 2048, 1024, 512, 256 that still gives every device two windows (so that uploads overlap the scoring)
        int64_t cap = ctx->shape_inflate_window > 0 ? ctx->shape_inflate_window : kShapeWindowInflate;
        while (cap > 256 && (uint64_t) cap * bytes > 0xFFFFFFFFull) cap /= 2;      // the strip table addresses a window's pixels with 32 bits
        for (int64_t w = cap; w >= 256; w /= 2)
            if ((int64_t) active.size() * 4 >= 7 * w * D) { win = w; break; }      // "two": the second may be three quarters full
    }
    const int64_t n_windows = ((int64_t) active.size() + win - 1) / win;
    const int used = (int) std::min<int64_t>(D, n_windows);

    // window w -> device w % used; per device the pairs of its windows in window order
    std::vector<ShapeDevWork> work(used);
    std::vector<std::vector<std::pair<int64_t, int64_t>>> win_pairs(used);      // per device and window: [first, end) into its pair arrays
    for (int64_t w = 0; w < n_windows; w++) {
        ShapeDevWork &wk = work[w % used];
        const int64_t a0 = w * win, a1 = std::min<int64_t>((int64_t) active.size(), a0 + win);
        const int64_t first = (int64_t) wk.pm.size();
        for (int64_t a = a0; a < a1; a++)
            for (int64_t q = tstart[active[a]]; q < tstart[active[a] + 1]; q++) {
                wk.pm.push_back(pair_mask[order[q]]);
                wk.ps.push_back((int32_t) (a - a0));
                wk.where.push_back(order[q]);
            }
        win_pairs[w % used].push_back({first, (int64_t) wk.pm.size()});
        wk.windows++;
    }

    std::vector<std::unique_ptr<PoolGuard>> guards;
    // files: one upload of the window's file bytes (run by run), ONE strip table and ONE decode launch per window; the tables go
    // through two pinned host slots per device
    size_t comp_cap = 0, strips_cap = 0;
    if (from_files) {
        for (int64_t w = 0; w < n_windows; w++) {
            size_t sum = 0;
            for (int64_t a = w * win; a < std::min<int64_t>((int64_t) active.size(), (w + 1) * win); a++) sum += (size_t) (offsets[active[a] + 1] - offsets[active[a]]);
            comp_cap = std::max(comp_cap, sum + 64);
        }
        strips_cap = (size_t) win * tiff_strips_bound(W, H);
    }
    // gradient images as PNG files: inflated scanlines of a window go through two pinned host slots per device
    const size_t png_stride = ((size_t) H * (1 + (size_t) W * 2) + 15) / 16 * 16;
    // device inflate: a slot holds the window's jobs, bytes per sample and zlib streams (the files are an upper bound of those), then
    // the statuses that come back; host inflate: the inflated scanlines
    const size_t z_head = ((size_t) win * (sizeof(InflateJob) + 1) + 15) / 16 * 16;
    size_t z_payload = 0;
    if (dev_inflate) {
        for (int64_t i = 0; i <= n_targets; i++)
            if (png_offsets[i] < 0 || (i > 0 && png_offsets[i] < png_offsets[i - 1])) return ctx->fail(CDS_ERR_BAD_ARG, "cds_shape_score_pairs_files: offsets must be non-decreasing");
        for (int64_t w = 0; w < n_windows; w++) {
            size_t sum = 0;
            for (int64_t a = w * win; a < std::min<int64_t>((int64_t) active.size(), (w + 1) * win); a++) sum += (size_t) (png_offsets[active[a] + 1] - png_offsets[active[a]]);
            z_payload = std::max(z_payload, sum + (size_t) 8 * win + 8);      // + alignment gaps
        }
        z_payload = (z_payload + 15) / 16 * 16;
        if (z_head + z_payload > 0xFFFFFFF0ull) return ctx->fail(CDS_ERR_UNSUPPORTED, "cds_shape_score_pairs_files: gradient files of one window exceed 4 GB");
    }
    const size_t z_stat = ((size_t) win * sizeof(int32_t) + 15) / 16 * 16;
    const size_t png_slot_bytes = dev_inflate ? z_head + z_payload + z_stat : (size_t) win * png_stride + (size_t) win;
    for (int d = 0; d < used; d++) {
        DevState &ds = ctx->devs[d];
        ShapeDevWork &wk = work[d];
        SH_CUDA(ctx, cudaSetDevice(ds.dev));
        SH_TRY(ensure_shape_tables(ctx, ds));
        cds_shape_maskset::Dev &sd = sms->dev[d];
        if (sd.dirty) {
            if (sd.d_descs_cap < sd.h_descs.size()) {
                SH_CUDA(ctx, cudaStreamSynchronize(ds.stream));
                if (sd.d_descs) { cudaFree(sd.d_descs); sd.d_descs = nullptr; sd.d_descs_cap = 0; }
                const size_t cap = std::max<size_t>(sd.h_descs.size() * 2, 64);
                SH_CUDA(ctx, cudaMalloc(&sd.d_descs, cap * sizeof(ShapeMaskDesc)));
                sd.d_descs_cap = cap;
            }
            SH_CUDA(ctx, cudaMemcpy(sd.d_descs, sd.h_descs.data(), sd.h_descs.size() * sizeof(ShapeMaskDesc), cudaMemcpyHostToDevice));
            sd.dirty = false;
        }
        guards.emplace_back(new PoolGuard(&ds));
        PoolGuard &g = *guards.back();
        // buffers come from the device's caching pool: consecutive calls (one per mask batch in gradientScores) reuse them
        for (int s = 0; s < 2; s++) {
            SH_CUDA(ctx, g.alloc((void **) &wk.d_t[s], win * bytes));
            SH_CUDA(ctx, g.alloc((void **) &wk.d_grad[s], win * px * sizeof(uint16_t)));
            if (zgap_rgb) SH_CUDA(ctx, g.alloc((void **) &wk.d_z[s], win * bytes));
        }
        SH_CUDA(ctx, g.alloc((void **) &wk.d_zslice, win * px * sizeof(uint16_t)));
        SH_CUDA(ctx, g.alloc((void **) &wk.d_tsig, win * bm_words * sizeof(uint32_t)));
        if (from_files) {
            SH_CUDA(ctx, g.alloc((void **) &wk.d_comp, comp_cap));
            SH_CUDA(ctx, g.alloc((void **) &wk.d_strips, strips_cap * sizeof(TiffStrip)));
            SH_TRY(ctx->ensure_pinned(ds, 2 * strips_cap * sizeof(TiffStrip)));
        }
        if (from_png) {
            SH_CUDA(ctx, g.alloc((void **) &wk.d_pngraw, (size_t) win * png_stride));
            SH_CUDA(ctx, g.alloc((void **) &wk.d_bps, (size_t) win));
            if (dev_inflate) {
                SH_CUDA(ctx, g.alloc((void **) &wk.d_zstage, z_head + z_payload));
                SH_CUDA(ctx, g.alloc((void **) &wk.d_zstat, z_stat));
                SH_CUDA(ctx, g.alloc((void **) &wk.d_zfallback, png_stride + 16));
            }
            if (ds.h_pinned2_bytes < 2 * png_slot_bytes) {
                SH_CUDA(ctx, cudaStreamSynchronize(ds.copy_stream));
                if (ds.h_pinned2) { cudaFreeHost(ds.h_pinned2); ds.h_pinned2 = nullptr; ds.h_pinned2_bytes = 0; }
                SH_CUDA(ctx, cudaHostAlloc(&ds.h_pinned2, 2 * png_slot_bytes, cudaHostAllocDefault));
                ds.h_pinned2_bytes = 2 * png_slot_bytes;
            }
        }
        const size_t np = wk.pm.size();
        SH_CUDA(ctx, g.alloc((void **) &wk.d_pm, np * sizeof(int32_t)));
        SH_CUDA(ctx, g.alloc((void **) &wk.d_ps, np * sizeof(int32_t)));
        SH_CUDA(ctx, g.alloc((void **) &wk.d_gap, np * sizeof(long long)));
        SH_CUDA(ctx, g.alloc((void **) &wk.d_he, np * sizeof(long long)));
        SH_CUDA(ctx, g.alloc((void **) &wk.d_mir, np));
        wk.h_gap.resize(np); wk.h_he.resize(np); wk.h_mir.resize(np);
        SH_CUDA(ctx, cudaStreamSynchronize(ds.stream));     // pooled buffers may still be in use by an earlier call
        SH_CUDA(ctx, cudaMemcpyAsync(wk.d_pm, wk.pm.data(), np * sizeof(int32_t), cudaMemcpyHostToDevice, ds.stream));
        SH_CUDA(ctx, cudaMemcpyAsync(wk.d_ps, wk.ps.data(), np * sizeof(int32_t), cudaMemcpyHostToDevice, ds.stream));
        while (ds.shape_timing.size() < (size_t) 2 * wk.windows) {
            cudaEvent_t e;
            SH_CUDA(ctx, cudaEventCreate(&e));
            ds.shape_timing.push_back(e);
        }
    }

    // Uploads (target, its gradient, its zgap image when given) of window j + 1 run on the copy stream while the main stream turns
    // window j into slice / signal planes and scores its pairs.  Runs of consecutive targets travel as one copy.
    std::vector<TiffStrip> strips;
    auto upload_window = [&](int d, int64_t j) -> cds_status {
        DevState &ds = ctx->devs[d];
        ShapeDevWork &wk = work[d];
        const int64_t w = j * used + d;
        const int slot = (int) (j & 1);
        const int64_t a0 = w * win, a1 = std::min<int64_t>((int64_t) active.size(), a0 + win);
        SH_CUDA(ctx, cudaSetDevice(ds.dev));
        if (j >= 2) SH_CUDA(ctx, cudaStreamWaitEvent(ds.copy_stream, ds.up_free[slot], 0));
        strips.clear();
        size_t comp_off = 0;
        for (int64_t a = a0; a < a1;) {
            int64_t e = a + 1;
            while (e < a1 && active[e] == active[e - 1] + 1) e++;
            const int64_t t0 = active[a], cnt = e - a, s0 = a - a0;
            if (from_files) {
                std::string err;
                for (int64_t i = 0; i < cnt; i++) {
                    const int64_t fa = offsets[t0 + i], fb = offsets[t0 + i + 1];
                    cds_status fs = tiff_collect_strips(blob + fa, (size_t) (fb - fa), W, H, (uint64_t) (comp_off + (size_t) (fa - offsets[t0])),
                                                        (uint64_t) (s0 + i) * bytes, strips, err);
                    if (fs != CDS_OK) return ctx->fail(fs, "cds_shape_score_pairs_tiff: file " + std::to_string(t0 + i) + ": " + err);
                }
                const size_t run_bytes = (size_t) (offsets[t0 + cnt] - offsets[t0]);
                if (comp_off + run_bytes > comp_cap || strips.size() > strips_cap) return ctx->fail(CDS_ERR_CAPACITY, "cds_shape_score_pairs_tiff: internal staging too small");
                SH_CUDA(ctx, cudaMemcpyAsync(wk.d_comp + comp_off, blob + offsets[t0], run_bytes, cudaMemcpyHostToDevice, ds.copy_stream));
                ctx->stats.h2d_bytes += (int64_t) run_bytes;
                comp_off += run_bytes;
            } else {
                SH_CUDA(ctx, cudaMemcpyAsync(wk.d_t[slot] + (size_t) s0 * bytes, target_rgb + (size_t) t0 * bytes, (size_t) cnt * bytes, cudaMemcpyHostToDevice, ds.copy_stream));
                ctx->stats.h2d_bytes += (int64_t) (cnt * bytes);
            }
            if (!from_png) {
                SH_CUDA(ctx, cudaMemcpyAsync(wk.d_grad[slot] + (size_t) s0 * px, gradient + (size_t) t0 * px, (size_t) cnt * px * sizeof(uint16_t), cudaMemcpyHostToDevice, ds.copy_stream));
                ctx->stats.h2d_bytes += (int64_t) (cnt * px * sizeof(uint16_t));
            }
            if (zgap_rgb) {
                SH_CUDA(ctx, cudaMemcpyAsync(wk.d_z[slot] + (size_t) s0 * bytes, zgap_rgb + (size_t) t0 * bytes, (size_t) cnt * bytes, cudaMemcpyHostToDevice, ds.copy_stream));
                ctx->stats.h2d_bytes += (int64_t) (cnt * bytes);
            }
            a = e;
        }
        if (j >= 2 && (from_files || from_png)) SH_CUDA(ctx, cudaEventSynchronize(ds.up_done[slot]));      // the slot's previous tables / scanlines have left the host
        if (dev_inflate) {
            // the window's gradient files cross PCIe as stored: the host only strings every file's IDAT payloads together
            uint8_t *h_slot = (uint8_t *) ds.h_pinned2 + (size_t) slot * png_slot_bytes;
            InflateJob *h_jobs = (InflateJob *) h_slot;
            uint8_t *h_bps = h_slot + (size_t) win * sizeof(InflateJob), *h_z = h_slot + z_head;
            const int64_t cnt = a1 - a0;
            size_t zo = 2;                                         // every stream starts 2 bytes before a 4-byte boundary: its deflate data (behind the zlib header) is aligned
            for (int64_t i = 0; i < cnt; i++) {
                const int64_t f = active[a0 + i];
                std::string err;
                size_t used_bytes = 0;
                cds_status ps = png_collect_idat(png_blob + png_offsets[f], (size_t) (png_offsets[f + 1] - png_offsets[f]), W, H, h_z + zo, z_payload - zo,
                                                 z_head + zo, &used_bytes, &h_jobs[i], &h_bps[i], err);
                if (ps != CDS_OK) return ctx->fail(ps, "cds_shape_score_pairs_files: file " + std::to_string(f) + ": " + err);
                zo = (zo + used_bytes + 1) / 4 * 4 + 2;
            }
            SH_CUDA(ctx, cudaMemcpyAsync(wk.d_zstage, h_slot, z_head + zo, cudaMemcpyHostToDevice, ds.copy_stream));
            ctx->stats.h2d_bytes += (int64_t) (z_head + zo);
            const uint8_t *d_bps_w = wk.d_zstage + (size_t) win * sizeof(InflateJob);
            launch_png_inflate(wk.d_zstage, (const InflateJob *) wk.d_zstage, cnt, wk.d_pngraw, png_stride, d_bps_w, W, H, wk.d_zstat, ds.copy_stream);
            SH_CUDA(ctx, cudaMemcpyAsync(h_slot + z_head + z_payload, wk.d_zstat, (size_t) cnt * sizeof(int32_t), cudaMemcpyDeviceToHost, ds.copy_stream));
            launch_png_unfilter(wk.d_pngraw, png_stride, d_bps_w, cnt, W, H, wk.d_grad[slot], ds.copy_stream);
            ctx->stats.kernel_launches += 2;
            SH_CUDA(ctx, cudaGetLastError());
        } else if (from_png) {
            // inflate this window's gradient files on host threads (the devices are busy with earlier windows meanwhile)
            uint8_t *h_f = (uint8_t *) ds.h_pinned2 + (size_t) slot * png_slot_bytes, *h_bps = h_f + (size_t) win * png_stride;
            const int64_t cnt = a1 - a0;
            SH_TRY(png_inflate_many(ctx, "cds_shape_score_pairs_files", png_blob, png_offsets, active.data() + a0, cnt, W, H, h_f, png_stride, h_bps));
            SH_CUDA(ctx, cudaMemcpyAsync(wk.d_pngraw, h_f, (size_t) cnt * png_stride, cudaMemcpyHostToDevice, ds.copy_stream));
            SH_CUDA(ctx, cudaMemcpyAsync(wk.d_bps, h_bps, (size_t) cnt, cudaMemcpyHostToDevice, ds.copy_stream));
            ctx->stats.h2d_bytes += (int64_t) (cnt * png_stride + cnt);
            launch_png_unfilter(wk.d_pngraw, png_stride, wk.d_bps, cnt, W, H, wk.d_grad[slot], ds.copy_stream);
            ctx->stats.kernel_launches++;
            SH_CUDA(ctx, cudaGetLastError());
        }
        if (from_files) {
            TiffStrip *h_tab = (TiffStrip *) ds.h_pinned + (size_t) slot * strips_cap;
            memcpy(h_tab, strips.data(), strips.size() * sizeof(TiffStrip));
            SH_CUDA(ctx, cudaMemcpyAsync(wk.d_strips, h_tab, strips.size() * sizeof(TiffStrip), cudaMemcpyHostToDevice, ds.copy_stream));
            ctx->stats.h2d_bytes += (int64_t) (strips.size() * sizeof(TiffStrip));
            launch_tiff_decode(wk.d_comp, wk.d_strips, (int64_t) strips.size(), wk.d_t[slot], ds.copy_stream);
            ctx->stats.kernel_launches++;
            SH_CUDA(ctx, cudaGetLastError());
        }
        SH_CUDA(ctx, cudaEventRecord(ds.up_done[slot], ds.copy_stream));
        return CDS_OK;
    };

    cds_status st = CDS_OK;
    for (int d = 0; d < used && st == CDS_OK; d++) st = upload_window(d, 0);
    int64_t max_windows = 0;
    for (int d = 0; d < used; d++) max_windows = std::max(max_windows, work[d].windows);
    for (int64_t j = 0; j < max_windows && st == CDS_OK; j++) {
        for (int d = 0; d < used && st == CDS_OK; d++) {
            ShapeDevWork &wk = work[d];
            if (j >= wk.windows) continue;
            DevState &ds = ctx->devs[d];
            if (j + 1 < wk.windows) st = upload_window(d, j + 1);
            if (st != CDS_OK) break;
            const int slot = (int) (j & 1);
            const int64_t w = j * used + d;
            const int64_t cnt = std::min<int64_t>((int64_t) active.size(), (w + 1) * win) - w * win;
            st = ctx->check(cudaSetDevice(ds.dev), "cudaSetDevice");
            if (st == CDS_OK) st = ctx->check(cudaStreamWaitEvent(ds.stream, ds.up_done[slot], 0), "wait");
            if (st != CDS_OK) break;
            if (dev_inflate) {
                // a stream the device's decoder refused is inflated by zlib on the host (which also decides whether the file is at fault);
                // its scanlines take the place of the device's on the main stream, before the window is scored
                st = ctx->check(cudaEventSynchronize(ds.up_done[slot]), "gradient inflate");
                const int32_t *h_stat = (const int32_t *) ((const uint8_t *) ds.h_pinned2 + (size_t) slot * png_slot_bytes + z_head + z_payload);
                for (int64_t i = 0; i < cnt && st == CDS_OK; i++) {
                    if (h_stat[i] == 0 && !(ctx->device_inflate == 2 && (i & 1))) continue;
                    const int64_t f = active[w * win + i];
                    std::vector<uint8_t> lines(png_stride + 16);
                    std::string err;
                    int depth = 16;
                    const cds_status ps = png_inflate(png_blob + png_offsets[f], (size_t) (png_offsets[f + 1] - png_offsets[f]), W, H, &depth, lines.data(), png_stride, err);
                    if (ps != CDS_OK) { st = ctx->fail(ps, "cds_shape_score_pairs_files: file " + std::to_string(f) + ": " + err); break; }
                    lines[png_stride] = (uint8_t) (depth / 8);
                    st = ctx->check(cudaMemcpyAsync(wk.d_zfallback, lines.data(), png_stride + 16, cudaMemcpyHostToDevice, ds.stream), "fallback scanlines H2D");
                    if (st == CDS_OK) launch_png_unfilter(wk.d_zfallback, png_stride, wk.d_zfallback + png_stride, 1, W, H, wk.d_grad[slot] + (size_t) i * px, ds.stream);
                    if (st == CDS_OK) st = ctx->check(cudaStreamSynchronize(ds.stream), "fallback unfilter");      // `lines` is pageable and about to go
                    ctx->stats.host_inflate_fallbacks++;
                }
                if (st != CDS_OK) break;
            }
            launch_shape_target_planes(sms, ds, wk.d_t[slot], zgap_rgb ? wk.d_z[slot] : nullptr, cnt, wk.d_zslice, wk.d_tsig, ds.stream);
            ctx->stats.kernel_launches++;
            const auto pr = win_pairs[d][j];
            cudaEventRecord(ds.shape_timing[2 * j], ds.stream);
            if (pr.second > pr.first) {
                shape_pair_kernel<<<(unsigned) (pr.second - pr.first), 256, 0, ds.stream>>>(sms->dev[d].d_descs, wk.d_pm + pr.first, wk.d_ps + pr.first,
                                                                                            wk.d_zslice, wk.d_grad[slot], wk.d_tsig, W, H, bpitch, sms->mirror,
                                                                                            wk.d_gap + pr.first, wk.d_he + pr.first, wk.d_mir + pr.first);
                ctx->stats.kernel_launches++;
                ctx->stats.match_kernel_launches++;
            }
            cudaEventRecord(ds.shape_timing[2 * j + 1], ds.stream);
            st = ctx->check(cudaGetLastError(), "shape kernels");
            if (st == CDS_OK) st = ctx->check(cudaEventRecord(ds.up_free[slot], ds.stream), "record");
        }
    }
    for (int d = 0; d < used && st == CDS_OK; d++) {
        DevState &ds = ctx->devs[d];
        ShapeDevWork &wk = work[d];
        const size_t np = wk.pm.size();
        st = ctx->check(cudaSetDevice(ds.dev), "cudaSetDevice");
        if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(wk.h_gap.data(), wk.d_gap, np * sizeof(long long), cudaMemcpyDeviceToHost, ds.stream), "gap D2H");
        if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(wk.h_he.data(), wk.d_he, np * sizeof(long long), cudaMemcpyDeviceToHost, ds.stream), "he D2H");
        if (st == CDS_OK) st = ctx->check(cudaMemcpyAsync(wk.h_mir.data(), wk.d_mir, np, cudaMemcpyDeviceToHost, ds.stream), "mirrored D2H");
    }
    double kernel_ms = 0;
    for (int d = 0; d < used && st == CDS_OK; d++) {
        DevState &ds = ctx->devs[d];
        ShapeDevWork &wk = work[d];
        st = ctx->check(cudaSetDevice(ds.dev), "cudaSetDevice");
        if (st == CDS_OK) st = ctx->check(cudaStreamSynchronize(ds.stream), "shape pairs");
        if (st != CDS_OK) break;
        double dev_ms = 0;
        for (int64_t j = 0; j < wk.windows; j++) {
            float ms = 0;
            cudaEventElapsedTime(&ms, ds.shape_timing[2 * j], ds.shape_timing[2 * j + 1]);
            dev_ms += ms;
        }
        kernel_ms = std::max(kernel_ms, dev_ms);
        for (size_t i = 0; i < wk.where.size(); i++) {
            gap_out[wk.where[i]] = wk.h_gap[i];
            high_expr_out[wk.where[i]] = wk.h_he[i];
            mirrored_out[wk.where[i]] = wk.h_mir[i];
        }
    }
    if (st == CDS_OK) {
        ctx->stats.match_kernel_ms = kernel_ms;
        ctx->stats.total_device_ms = kernel_ms;
        ctx->stats.comparisons = n_pairs;
        ctx->stats.d2h_bytes = n_scored * 17;
    }
    return st;      // the guards drain both streams of every device before the pooled buffers go back
}

extern "C" cds_status cds_shape_score_pairs(cds_ctx *ctx, const cds_shape_maskset *sms, const uint8_t *target_rgb, const uint16_t *gradient,
                                            const uint8_t *zgap_rgb, const uint8_t *has_variants, int64_t n_targets,
                                            const int32_t *pair_mask, const int64_t *pair_target, int64_t n_pairs,
                                            int64_t *gap_out, int64_t *high_expr_out, uint8_t *mirrored_out)
{
    return cds::abi_guard("cds_shape_score_pairs", [&]() -> cds_status {
        return shape_score_pairs_impl(ctx, sms, target_rgb, nullptr, nullptr, gradient, nullptr, nullptr, zgap_rgb, has_variants, n_targets, pair_mask, pair_target, n_pairs,
                                      gap_out, high_expr_out, mirrored_out);
    });
}

extern "C" cds_status cds_shape_score_pairs_tiff(cds_ctx *ctx, const cds_shape_maskset *sms, const uint8_t *blob, const int64_t *offsets,
                                                 const uint16_t *gradient, const uint8_t *zgap_rgb, const uint8_t *has_variants, int64_t n_targets,
                                                 const int32_t *pair_mask, const int64_t *pair_target, int64_t n_pairs,
                                                 int64_t *gap_out, int64_t *high_expr_out, uint8_t *mirrored_out)
{
    return cds::abi_guard("cds_shape_score_pairs_tiff", [&]() -> cds_status {
        if (n_targets > 0 && (!blob || !offsets)) { set_tls_error("cds_shape_score_pairs_tiff: NULL files"); return CDS_ERR_BAD_ARG; }
        return shape_score_pairs_impl(ctx, sms, nullptr, blob, offsets, gradient, nullptr, nullptr, zgap_rgb, has_variants, n_targets, pair_mask, pair_target, n_pairs,
                                      gap_out, high_expr_out, mirrored_out);
    });
}

extern "C" cds_status cds_shape_score_pairs_files(cds_ctx *ctx, const cds_shape_maskset *sms, const uint8_t *tiff_blob, const int64_t *tiff_offsets,
                                                  const uint8_t *png_blob, const int64_t *png_offsets, const uint8_t *zgap_rgb,
                                                  const uint8_t *has_variants, int64_t n_targets,
                                                  const int32_t *pair_mask, const int64_t *pair_target, int64_t n_pairs,
                                                  int64_t *gap_out, int64_t *high_expr_out, uint8_t *mirrored_out)
{
    return cds::abi_guard("cds_shape_score_pairs_files", [&]() -> cds_status {
        if (n_targets > 0 && (!tiff_blob || !tiff_offsets || !png_blob || !png_offsets)) { set_tls_error("cds_shape_score_pairs_files: NULL files"); return CDS_ERR_BAD_ARG; }
        return shape_score_pairs_impl(ctx, sms, nullptr, tiff_blob, tiff_offsets, nullptr, png_blob, png_offsets, zgap_rgb, has_variants, n_targets,
                                      pair_mask, pair_target, n_pairs, gap_out, high_expr_out, mirrored_out);
    });
}

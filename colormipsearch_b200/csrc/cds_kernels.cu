// cds_kernels.cu -- library encoding, mask preparation and the generic (any xyShift) pixel-match kernel.
//
// Reference semantics (API/ = colormipsearch-api/src/main/java/org/janelia/colormipsearch/):
//   encode        : the target side of calculatePixelGap, API/cds/AbstractColorDepthSearchAlgorithm.java:225-257, folded
//                   into the integer code word described in cds_common.h
//   mask records  : getMaskPosArray, API/cds/AbstractColorDepthSearchAlgorithm.java:96-126 (+ the mask side of calculatePixelGap)
//   gather kernel : calculateScore / calculateMaxScoreForAllTargetTransformations / calculateMatchingScore,
//                   API/cds/PixelMatchColorDepthSearchAlgorithm.java:166-263, with the shifted / mirrored position lists of
//                   :113-158 evaluated on the fly instead of being materialised.
#include "cds_kernels.cuh"

namespace cds {

// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int classify_color_dev(int r, int g, int b, int &second, int &maxv)
{
    if (b > r && b > g) { maxv = b; if (r > g) { second = r; return 0; } second = g; return 1; }
    if (g > b && g > r) { maxv = g; if (b > r) { second = b; return 2; } second = r; return 3; }
    if (r > b && r > g) { maxv = r; if (g > b) { second = g; return 4; } second = b; return 5; }
    maxv = max(r, max(g, b));
    second = 0;
    return -1;
}

__device__ __forceinline__ uint32_t encode_color_dev(int r, int g, int b, const uint16_t *__restrict__ rank_tab, int thr)
{
    int second, maxv;
    int sector = classify_color_dev(r, g, b, second, maxv);
    uint32_t sr = sector < 0 ? (uint32_t) CDS_SR_NONE
                             : (uint32_t) sector * CDS_SECTOR_STRIDE + __ldg(rank_tab + second * 256 + maxv);
    uint32_t code = (sr << CDS_CODE_SR_SHIFT) | (uint32_t) maxv;
    if (!(maxv > thr)) code |= CDS_CODE_BELOW_BIT;
    return code;
}

__global__ void fill_words_kernel(uint32_t *__restrict__ p, size_t n, uint32_t v)
{
    size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t) gridDim.x * blockDim.x;
    // 128-bit stores on the aligned body
    size_t n4 = n / 4;
    uint4 v4 = make_uint4(v, v, v, v);
    uint4 *p4 = reinterpret_cast<uint4 *>(p);
    for (size_t k = i; k < n4; k += stride) p4[k] = v4;
    for (size_t k = n4 * 4 + i; k < n; k += stride) p[k] = v;
}

void launch_fill_words(uint32_t *p, size_t n, uint32_t v, cudaStream_t s)
{
    if (n == 0) return;
    fill_words_kernel<<<148 * 8, 256, 0, s>>>(p, n, v);
}

// One CTA per (image row, image).  The RGB row (3W bytes, arbitrary alignment) is staged through shared memory with
// aligned 32-bit loads; each warp then encodes 32 consecutive pixels per iteration and writes coalesced code words, pads
// included.  With VALID the kernel also emits the row's per-sector "can match" bits (what valid_bits_kernel derives from
// the code words) while the pixels are in registers: six ballots per 32 pixels instead of a second pass over the planes.
__device__ __forceinline__ int code_sector(uint32_t cw)
{
    // above the threshold, and in a colour sector: "no sector" pixels (ties for the maximum, e.g. grey) have pixel gap
    // 10000 against everything (AbstractColorDepthSearchAlgorithm.java:182, 259-388), they can never match
    const uint32_t sr = (cw >> CDS_CODE_SR_SHIFT) & 0x3FFFFu;
    if ((cw & (CDS_CODE_BELOW_BIT | CDS_CODE_PAD_BIT)) == 0 && sr < (uint32_t) CDS_SR_NONE) return (int) (sr / CDS_SECTOR_STRIDE);
    return -1;
}

constexpr int kEncodeRows = 4;      // image rows per CTA (fewer for very wide images): one staging round trip to DRAM per 4 rows
constexpr int kEncodeQueue = 64;    // per-warp queue of non-black pixels waiting for the colour classifier (power of two, >= 2 * 32)

template <bool VALID>
__global__ void __launch_bounds__(256) encode_rgb_kernel(const uint8_t *__restrict__ rgb, uint32_t *__restrict__ planes, PlaneGeom g,
                                                         int64_t first_slot, const uint16_t *__restrict__ rank_tab, int thr,
                                                         int vp, uint32_t *__restrict__ valid /* chunk-relative [n][H][sectors][vp] */,
                                                         int rows_per_cta)
{
    extern __shared__ uint4 srow4[];
    const int y0 = blockIdx.x * rows_per_cta;
    const int rows = min(rows_per_cta, g.H - y0);
    const int64_t img = blockIdx.y;
    const size_t row_bytes = (size_t) g.W * 3;
    // the rows are contiguous in the source: stage them with aligned 128-bit loads (the source has arbitrary alignment)
    const uint8_t *src = rgb + ((size_t) img * g.H + y0) * row_bytes;
    const uintptr_t a = reinterpret_cast<uintptr_t>(src);
    const int off = (int) (a & 15);
    const uint4 *asrc = reinterpret_cast<const uint4 *>(a - off);
    const int n_vec = (int) ((off + rows * row_bytes + 15) / 16);
    for (int k = threadIdx.x; k < n_vec; k += blockDim.x) srow4[k] = asrc[k];
    const uint8_t *sb = reinterpret_cast<const uint8_t *>(srow4) + off;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int kmax = (g.pitch + 31) >> 5;
    // the rows' valid words are collected behind the staged pixels and leave as one contiguous block: a lane writing single
    // words at a stride of vp makes every store a partial-sector write that L2 has to merge
    uint32_t *s_valid = reinterpret_cast<uint32_t *>(srow4 + (rows_per_cta * row_bytes + 15 + 15) / 16);
    uint32_t *s_queue = s_valid + (VALID ? rows_per_cta * CDS_NUM_SECTORS * vp : 0);       // [warps][kEncodeQueue] pixels to encode
    if (VALID)
        for (int k = threadIdx.x; k < rows * CDS_NUM_SECTORS * vp; k += blockDim.x) s_valid[k] = 0u;
    __syncthreads();
    // Colour-depth MIPs are mostly black (~94 % of the pixels): black pixels get the black code word straight away, and only the
    // others run the colour classifier (~150 instructions) -- compacted warp-wide into a small queue so that the classifier always
    // runs on full warps.  Work is proportional to the non-black pixels, not to the 32-pixel groups that contain one.
    const uint32_t black = encode_color_dev(0, 0, 0, rank_tab, thr);
    uint32_t *prow0 = planes + g.row_offset(first_slot + img, y0);
    uint32_t *myq = s_queue + warp * kEncodeQueue;
    const uint32_t lt = (1u << lane) - 1u;
    uint32_t qh = 0, qt = 0;
    auto drain = [&](bool all) {
        while (qt - qh >= 32u || (all && qt != qh)) {
            const uint32_t n = min(32u, qt - qh);
            if ((uint32_t) lane < n) {
                const uint32_t e = myq[(qh + lane) & (kEncodeQueue - 1)];
                const int x = (int) (e & 0xFFFFu), r = (int) (e >> 16);
                const uint8_t *px = sb + (size_t) r * row_bytes + 3 * x;
                const uint32_t code = encode_color_dev(px[0], px[1], px[2], rank_tab, thr);
                prow0[(size_t) r * g.pitch + x] = code;
                if (VALID) {
                    const int sector = code_sector(code);
                    if (sector >= 0) atomicOr(&s_valid[(r * CDS_NUM_SECTORS + sector) * vp + (x >> 5)], 1u << (x & 31));
                }
            }
            qh += n;
            __syncwarp();
        }
    };
    for (int r = 0; r < rows; r++) {
        uint32_t *drow = prow0 + (size_t) r * g.pitch;
        const uint8_t *srow = sb + (size_t) r * row_bytes;
        for (int k = warp; k < kmax; k += (int) (blockDim.x >> 5)) {
            const int x = k * 32 + lane;
            bool lit = false;
            if (x < g.W) lit = (srow[3 * x] | srow[3 * x + 1] | srow[3 * x + 2]) != 0;
            if (x < g.pitch && !lit) drow[x] = x < g.W ? black : CDS_CODE_PAD_WORD;
            const unsigned m = __ballot_sync(0xffffffffu, lit);
            if (m) {
                if (lit) myq[(qt + (uint32_t) __popc(m & lt)) & (kEncodeQueue - 1)] = (uint32_t) x | ((uint32_t) r << 16);
                qt += (uint32_t) __popc(m);
                __syncwarp();
                drain(false);
            }
        }
    }
    drain(true);
    if (VALID) {
        __syncthreads();
        uint32_t *vout = valid + ((size_t) img * g.H + y0) * CDS_NUM_SECTORS * vp;
        for (int k = threadIdx.x; k < rows * CDS_NUM_SECTORS * vp; k += blockDim.x) vout[k] = s_valid[k];
    }
}

void launch_encode_rgb(const uint8_t *rgb, int64_t n, uint32_t *planes, PlaneGeom g, int64_t first_slot,
                       const uint16_t *rank_tab, int data_threshold, cudaStream_t s, uint32_t *valid)
{
    if (n == 0) return;
    const int vp = occupancy_valid_pitch(g.W);
    int rpc = kEncodeRows;
    auto smem_for = [&](int r) { return ((size_t) r * g.W * 3 + 15 + 15) / 16 * 16 + (valid ? (size_t) r * CDS_NUM_SECTORS * vp * 4 : 0) + (size_t) 8 * kEncodeQueue * 4; };
    while (rpc > 1 && smem_for(rpc) > 96 * 1024) rpc >>= 1;
    const size_t smem = smem_for(rpc);
    static bool attr_set = false;
    if (!attr_set) {
        // wide images need more than the default 48 kB of dynamic shared memory
        cudaFuncSetAttribute(encode_rgb_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(encode_rgb_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        attr_set = true;
    }
    // gridDim.y is limited to 65535: chunk
    for (int64_t i0 = 0; i0 < n; i0 += 32768) {
        int64_t cnt = n - i0 < 32768 ? n - i0 : 32768;
        dim3 grid((g.H + rpc - 1) / rpc, (unsigned) cnt);
        const uint8_t *src = rgb + (size_t) i0 * g.H * g.W * 3;
        if (valid)
            encode_rgb_kernel<true><<<grid, 256, smem, s>>>(src, planes, g, first_slot + i0, rank_tab, data_threshold, vp,
                                                            valid + (size_t) i0 * g.H * CDS_NUM_SECTORS * vp, rpc);
        else
            encode_rgb_kernel<false><<<grid, 256, smem, s>>>(src, planes, g, first_slot + i0, rank_tab, data_threshold, vp, nullptr, rpc);
    }
}

__global__ void rebake_kernel(uint32_t *__restrict__ p, size_t n, int thr)
{
    size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t) gridDim.x * blockDim.x;
    size_t n4 = n / 4;
    uint4 *p4 = reinterpret_cast<uint4 *>(p);
    auto bake = [thr](uint32_t c) -> uint32_t {
        if (c & CDS_CODE_PAD_BIT) return c;
        uint32_t below = ((int) (c & 0xFFu) > thr) ? 0u : CDS_CODE_BELOW_BIT;
        return (c & ~CDS_CODE_BELOW_BIT) | below;
    };
    for (size_t k = i; k < n4; k += stride) {
        uint4 v = p4[k];
        v.x = bake(v.x); v.y = bake(v.y); v.z = bake(v.z); v.w = bake(v.w);
        p4[k] = v;
    }
    for (size_t k = n4 * 4 + i; k < n; k += stride) p[k] = bake(p[k]);
}

void launch_rebake(uint32_t *planes, size_t n_words, int data_threshold, cudaStream_t s)
{
    if (n_words == 0) return;
    rebake_kernel<<<148 * 8, 256, 0, s>>>(planes, n_words, data_threshold);
}

__global__ void encode_colors_kernel(const uint8_t *__restrict__ rgb, int64_t n, const uint16_t *__restrict__ rank_tab, int thr,
                                     uint32_t *__restrict__ codes)
{
    int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t) gridDim.x * blockDim.x;
    for (; i < n; i += stride) codes[i] = encode_color_dev(rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2], rank_tab, thr);
}

void launch_encode_colors(const uint8_t *rgb, int64_t n, const uint16_t *rank_tab, int data_threshold, uint32_t *codes, cudaStream_t s)
{
    if (n == 0) return;
    encode_colors_kernel<<<148 * 4, 256, 0, s>>>(rgb, n, rank_tab, data_threshold, codes);
}

// ------------------------------------------------------------------------------------------------------------------
// Occupancy bitmaps (see cds_kernels.cuh).  Pass 1: per colour sector one bit per pixel "inside the image, above the
// threshold, in this sector"; pass 2: OR of the bits at the shift offsets, 32 pixels at a time with word shifts, plus the
// OR over the sectors in slot CDS_NUM_SECTORS.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) valid_bits_kernel(const uint32_t *__restrict__ planes, PlaneGeom g, int64_t t0, int vp,
                                                         uint32_t *__restrict__ valid /* chunk-relative [n][H][sectors][vp] */)
{
    extern __shared__ uint32_t s_valid[];
    const int y = blockIdx.x;
    const int64_t t = t0 + blockIdx.y;
    const uint32_t *row = planes + g.row_offset(t, y);
    uint32_t *out = valid + ((size_t) blockIdx.y * g.H + y) * CDS_NUM_SECTORS * vp;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = warp; k < vp; k += (int) (blockDim.x >> 5)) {
        const int x = k * 32 + lane;
        const int sector = x < g.W ? code_sector(row[x]) : -1;
#pragma unroll
        for (int s = 0; s < CDS_NUM_SECTORS; s++) {
            const unsigned bal = __ballot_sync(0xffffffffu, sector == s);
            if (lane == 0) s_valid[s * vp + k] = bal;
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < CDS_NUM_SECTORS * vp; k += blockDim.x) out[k] = s_valid[k];      // one contiguous block per row
}

__device__ __forceinline__ uint32_t hspread(const uint32_t *__restrict__ vrow, int k, int vp, int s)
{
    // bit x of the result = valid(x - s) | valid(x) | valid(x + s)
    const uint32_t c = vrow[k];
    const uint32_t l = k > 0 ? vrow[k - 1] : 0u;
    const uint32_t r = k + 1 < vp ? vrow[k + 1] : 0u;
    return c | (c << s) | (l >> (32 - s)) | (c >> s) | (r << (32 - s));
}

// One thread per 32-pixel strip of one TILE row (4 image rows): per sector the dilated bits of the four rows, transposed
// into the strip's four 8 x 4 tile words and written as one 128-bit store -- consecutive threads write consecutive 16 bytes.
template <int RINGS>
__device__ __forceinline__ void occupancy_strip(const uint32_t *__restrict__ vsec /* sector's words of row 0 */, int vrow_words, int H,
                                                int vp, int k, int y0, uint32_t o[4])
{
    if constexpr (RINGS == 0) {
#pragma unroll
        for (int r = 0; r < 4; r++) o[r] = y0 + r < H ? vsec[(size_t) (y0 + r) * vrow_words + k] : 0u;
        return;
    } else {
    uint32_t h2[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int y = y0 - 2 + j;
        h2[j] = (y >= 0 && y < H) ? hspread(vsec + (size_t) y * vrow_words, k, vp, 2) : 0u;
    }
#pragma unroll
    for (int r = 0; r < 4; r++) o[r] = h2[r] | h2[r + 2] | h2[r + 4];
    if (RINGS >= 2) {
        uint32_t h4[12];
#pragma unroll
        for (int j = 0; j < 12; j++) {
            const int y = y0 - 4 + j;
            h4[j] = (y >= 0 && y < H) ? hspread(vsec + (size_t) y * vrow_words, k, vp, 4) : 0u;
        }
#pragma unroll
        for (int r = 0; r < 4; r++) o[r] |= h4[r] | h4[r + 4] | h4[r + 8];
    }
#pragma unroll
    for (int r = 0; r < 4; r++) if (y0 + r >= H) o[r] = 0u;       // rows of the last tile row that lie below the image
    }
}

// rows o[0..3] of a 32-pixel strip -> its four tile words (byte r of word j = byte j of row r)
__device__ __forceinline__ uint4 strip_to_tiles(const uint32_t o[4])
{
    const uint32_t a = __byte_perm(o[0], o[1], 0x5140), b = __byte_perm(o[2], o[3], 0x5140);
    const uint32_t c = __byte_perm(o[0], o[1], 0x7362), d = __byte_perm(o[2], o[3], 0x7362);
    return make_uint4(__byte_perm(a, b, 0x5410), __byte_perm(a, b, 0x7632), __byte_perm(c, d, 0x5410), __byte_perm(c, d, 0x7632));
}

template <int RINGS>
__global__ void __launch_bounds__(256) occupancy_kernel(const uint32_t *__restrict__ valid /* chunk-relative */, int H, int vp, int tp,
                                                        int64_t t0, int64_t n, uint32_t *__restrict__ occ)
{
    const int rowpitch = occupancy_row_pitch(tp);
    const int HT = occupancy_tile_rows(H);
    const int vrow_words = CDS_NUM_SECTORS * vp;
    const size_t total = (size_t) n * HT * vp;
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
        const int k = (int) (i % vp);
        const int ty = (int) ((i / vp) % HT);
        const int64_t tl = (int64_t) (i / ((size_t) vp * HT));
        if (4 * k >= tp) continue;                     // tp is a multiple of 4: a strip is four whole tile words or none
        const uint32_t *vimg = valid + (size_t) tl * H * vrow_words;
        uint32_t *trow = occ + ((size_t) (t0 + tl) * HT + ty) * rowpitch;
        uint4 *orow = reinterpret_cast<uint4 *>(trow) + k;
        uint32_t *nz = trow + occupancy_nz_offset(tp);          // the row's non-empty bits: zero on entry (launch_occupancy_kernel clears them)
        uint32_t any[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int s = 0; s < CDS_NUM_SECTORS; s++) {
            uint32_t o[4];
            occupancy_strip<RINGS>(vimg + s * vp, vrow_words, H, vp, k, 4 * ty, o);
#pragma unroll
            for (int r = 0; r < 4; r++) any[r] |= o[r];
            const uint4 t = strip_to_tiles(o);
            orow[(size_t) s * (tp / 4)] = t;
            // one bit per sector tile word, "this word is not empty": bit s * tp + 4 k + j for the strip's four words (the four bits never
            // straddle a 32-bit word: tp and 4 k are multiples of 4).  Occupied tiles are few, so this is a rare atomic, not a second pass.
            const uint32_t nib = (t.x != 0u ? 1u : 0u) | (t.y != 0u ? 2u : 0u) | (t.z != 0u ? 4u : 0u) | (t.w != 0u ? 8u : 0u);
            if (nib) {
                const int bit = s * tp + 4 * k;
                atomicOr(&nz[bit >> 5], nib << (bit & 31));
            }
        }
        reinterpret_cast<uint4 *>(trow + occupancy_any_offset(tp))[k] = strip_to_tiles(any);
    }
}

// The same for xyShift 2 (the production setting), every valid word read ONCE: a thread owns one 32-pixel column of one target and
// walks down a segment of kOccSegRows tile rows with the last four image rows of every sector in registers, so a tile row costs four
// new rows per sector instead of eight, and the vertical OR (rows y - 2, y, y + 2) is done on the raw words BEFORE the horizontal
// spread (both are ORs of shifted copies, so they commute) -- four spreads per sector instead of eight.  The spread needs the
// neighbouring columns' words: the threads of a block exchange them through shared memory (zero columns on both sides).
constexpr int kOccThreads = 256;
constexpr int kOccSegRows = 12;

__global__ void __launch_bounds__(kOccThreads) occupancy_ring1_kernel(const uint32_t *__restrict__ valid /* chunk-relative */, int H, int vp, int tp,
                                                                      int64_t t0, uint32_t *__restrict__ occ, int segs, int blocks_per_target)
{
    extern __shared__ uint32_t s_v[];                     // [sector][row of the tile][segment][kc + 2]
    const int kc = tp / 4;                                // 32-pixel columns that hold tile words
    const int cw = kc + 2;
    const int seg = (int) threadIdx.x / kc, k = (int) threadIdx.x - seg * kc;
    const int rowpitch = occupancy_row_pitch(tp);
    const int HT = occupancy_tile_rows(H);
    const int vrow_words = CDS_NUM_SECTORS * vp;
    const int64_t tl = blockIdx.x / blocks_per_target;
    const int ty0 = ((int) (blockIdx.x % blocks_per_target) * segs + seg) * kOccSegRows;
    const bool active = seg < segs && ty0 < HT;
    const uint32_t *vimg = valid + (size_t) tl * H * vrow_words + k;
    auto sv = [&](int s, int r) -> uint32_t * { return s_v + ((s * 4 + r) * segs + seg) * cw; };
    if (seg < segs && (k == 0 || k == kc - 1))
        for (int i = 0; i < CDS_NUM_SECTORS * 4; i++) (s_v + (i * segs + seg) * cw)[k == 0 ? 0 : kc + 1] = 0u;
    if (seg < segs && kc == 1)
        for (int i = 0; i < CDS_NUM_SECTORS * 4; i++) (s_v + (i * segs + seg) * cw)[0] = 0u;
    auto raw = [&](int s, int y) -> uint32_t { return (active && y >= 0 && y < H) ? __ldg(vimg + (size_t) y * vrow_words + s * vp) : 0u; };
    // the tile row's non-empty bits are collected in shared memory and leave as plain stores: no clearing pass over the rows beforehand,
    // no atomics on global memory (word i of a segment's row is written, read and cleared by the same thread)
    const int nzw = occupancy_nz_words(tp);
    uint32_t *s_nz = s_v + (size_t) CDS_NUM_SECTORS * 4 * segs * cw + (size_t) (seg < segs ? seg : 0) * nzw;
    uint32_t carry[CDS_NUM_SECTORS][4];                   // image rows y0 - 2 .. y0 + 1 of the coming tile row
#pragma unroll
    for (int s = 0; s < CDS_NUM_SECTORS; s++)
#pragma unroll
        for (int j = 0; j < 4; j++) carry[s][j] = raw(s, 4 * ty0 - 2 + j);
    for (int it = 0; it < kOccSegRows; it++) {
        const int ty = ty0 + it, y0 = 4 * ty;
        uint32_t nw[CDS_NUM_SECTORS][4];                  // rows y0 + 2 .. y0 + 5
#pragma unroll
        for (int s = 0; s < CDS_NUM_SECTORS; s++)
#pragma unroll
            for (int j = 0; j < 4; j++) nw[s][j] = raw(s, y0 + 2 + j);
        if (seg < segs) {
            for (int i = k; i < nzw; i += kc) s_nz[i] = 0u;
#pragma unroll
            for (int s = 0; s < CDS_NUM_SECTORS; s++) {
                sv(s, 0)[k + 1] = carry[s][0] | carry[s][2] | nw[s][0];
                sv(s, 1)[k + 1] = carry[s][1] | carry[s][3] | nw[s][1];
                sv(s, 2)[k + 1] = carry[s][2] | nw[s][0] | nw[s][2];
                sv(s, 3)[k + 1] = carry[s][3] | nw[s][1] | nw[s][3];
#pragma unroll
                for (int j = 0; j < 4; j++) carry[s][j] = nw[s][j];
            }
        }
        __syncthreads();
        if (active && ty < HT) {
            uint32_t *trow = occ + ((size_t) (t0 + tl) * HT + ty) * rowpitch;
            uint4 *orow = reinterpret_cast<uint4 *>(trow) + k;
            uint32_t any[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int s = 0; s < CDS_NUM_SECTORS; s++) {
                uint32_t o[4];
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    const uint32_t *v = sv(s, r) + k;
                    const uint32_t l = v[0], c = v[1], rr = v[2];
                    o[r] = y0 + r < H ? (c | (c << 2) | (c >> 2) | (l >> 30) | (rr << 30)) : 0u;
                    any[r] |= o[r];
                }
                const uint4 t = strip_to_tiles(o);
                orow[(size_t) s * (tp / 4)] = t;
                const uint32_t nib = (t.x != 0u ? 1u : 0u) | (t.y != 0u ? 2u : 0u) | (t.z != 0u ? 4u : 0u) | (t.w != 0u ? 8u : 0u);
                if (nib) {
                    const int bit = s * tp + 4 * k;
                    atomicOr(&s_nz[bit >> 5], nib << (bit & 31));
                }
            }
            reinterpret_cast<uint4 *>(trow + occupancy_any_offset(tp))[k] = strip_to_tiles(any);
        }
        __syncthreads();
        if (active && ty < HT) {
            uint32_t *nz = occ + ((size_t) (t0 + tl) * HT + ty) * rowpitch + occupancy_nz_offset(tp);
            for (int i = k; i < nzw; i += kc) nz[i] = s_nz[i];
        }
    }
}

int &occupancy_kernel_version()
{
    static int v = 1;       // 1: occupancy_ring1_kernel for xyShift 2; 0: the generic kernel everywhere (cross-check)
    return v;
}

static void launch_occupancy_kernel(const uint32_t *valid, int H, int vp, int tp, int64_t t0, int64_t n, int rings, uint32_t *occ, cudaStream_t s)
{
    // the non-empty bits behind every tile row start from zero: one strided clear instead of the separate pass that used to read every
    // tile word back (occupancy_nz_kernel, 0.26 ms per 1 024 targets)
    const int rowpitch = occupancy_row_pitch(tp);
    const int HT = occupancy_tile_rows(H);
    const int kc = tp / 4;
    if (rings == 1 && occupancy_kernel_version() == 1 && kc >= 1 && kc <= kOccThreads / 2 && n * 64 < (1ll << 31)) {
        const int segs = std::min(kOccThreads / kc, 8);          // segments per block; keeps the exchange buffer below 32 kB
        const int blocks_per_target = (HT + segs * kOccSegRows - 1) / (segs * kOccSegRows);
        const size_t smem = ((size_t) CDS_NUM_SECTORS * 4 * segs * (kc + 2) + (size_t) segs * occupancy_nz_words(tp)) * sizeof(uint32_t);
        occupancy_ring1_kernel<<<(unsigned) (n * blocks_per_target), kOccThreads, smem, s>>>(valid, H, vp, tp, t0, occ, segs, blocks_per_target);
        return;
    }
    // the generic kernel ORs its non-empty bits into rows that start from zero: one strided clear
    cudaMemset2DAsync(occ + (size_t) t0 * HT * rowpitch + (size_t) occupancy_nz_offset(tp), (size_t) rowpitch * sizeof(uint32_t), 0,
                      (size_t) occupancy_nz_words(tp) * sizeof(uint32_t), (size_t) n * HT, s);
    if (rings == 0) occupancy_kernel<0><<<148 * 8, 256, 0, s>>>(valid, H, vp, tp, t0, n, occ);
    else if (rings == 1) occupancy_kernel<1><<<148 * 8, 256, 0, s>>>(valid, H, vp, tp, t0, n, occ);
    else occupancy_kernel<2><<<148 * 8, 256, 0, s>>>(valid, H, vp, tp, t0, n, occ);
}

// Rank-band bytes (cds_kernels.cuh).  One CTA per (target, tile row).  The per-sector valid bits that the occupancy kernels read say which
// pixels of the rows [4 ty - S, 4 ty + 3 + S] count (in the image, above the baked threshold, of that sector; a few per cent of them), so
// only those pixels' code words are read, for their ranks; their band bits (sector * 8 + band, 48 of them) are ORed per column in shared
// memory.  Then every tile ORs the columns [8 tx - S, 8 tx + 7 + S], and the bytes leave as whole words.
constexpr int kBandThreads = 256;
constexpr int kBandPad = 4;                                // >= the largest xyShift
static_assert(CDS_NUM_SECTORS * CDS_RANK_BANDS <= 64, "a column's band bits are one 64-bit word");

__global__ void __launch_bounds__(kBandThreads) occupancy_bands_kernel(const uint32_t *__restrict__ valid /* chunk-relative */, int vp,
                                                                       const uint32_t *__restrict__ planes, PlaneGeom g, int64_t t0, int S,
                                                                       int tp, uint32_t *__restrict__ occ)
{
    extern __shared__ unsigned long long s_col[];          // [kBandPad + tp * 8 + kBandPad] column bits, then [tp] tile bits
    const int ty = blockIdx.x, HT = gridDim.x;
    const int64_t tl = blockIdx.y, t = t0 + tl;
    const int ncol = tp * 8;
    unsigned long long *s_tile = s_col + ncol + 2 * kBandPad;
    for (int i = threadIdx.x; i < ncol + 2 * kBandPad; i += kBandThreads) s_col[i] = 0ull;
    __syncthreads();
    const int ya = max(4 * ty - S, 0), yb = min(4 * ty + 3 + S, g.H - 1);
    const uint32_t *plane = planes + g.row_offset(t, 0);
    const int n_words = (yb - ya + 1) * vp;
    for (int i = threadIdx.x; i < n_words; i += kBandThreads) {
        const int y = ya + i / vp, k = i % vp;
        const uint32_t *vw = valid + ((size_t) tl * g.H + y) * CDS_NUM_SECTORS * vp + k;
#pragma unroll
        for (int sec = 0; sec < CDS_NUM_SECTORS; sec++) {
            uint32_t m = __ldg(vw + sec * vp);
            while (m) {
                const int x = 32 * k + __ffs((int) m) - 1;
                m &= m - 1u;
                if (x >= g.W) break;
                const uint32_t rank = (__ldg(plane + (size_t) y * g.pitch + x) >> CDS_CODE_SR_SHIFT) % CDS_SECTOR_STRIDE;
                atomicOr(&s_col[x + kBandPad], 1ull << (sec * CDS_RANK_BANDS + (int) occupancy_rank_band(rank)));
            }
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < tp; k += kBandThreads) {
        unsigned long long b = 0ull;
        for (int x = 8 * k - S; x <= 8 * k + 7 + S; x++) b |= s_col[x + kBandPad];
        s_tile[k] = b;
    }
    __syncthreads();
    uint32_t *out = occ + ((size_t) t * HT + ty) * occupancy_row_pitch(tp) + occupancy_band_offset(tp);
    const int nbw = occupancy_band_words(tp);
    for (int w = threadIdx.x; w < nbw; w += kBandThreads) {
        uint32_t v = 0u;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int i = 4 * w + j;                       // sector tile word i = sector * tp + tile column
            if (i < CDS_NUM_SECTORS * tp) v |= (uint32_t) ((s_tile[i % tp] >> (CDS_RANK_BANDS * (i / tp))) & 0xFFull) << (8 * j);
        }
        out[w] = v;
    }
}

// targets [t0, t0 + n), whose valid bits are targets [0, n) of `valid`
static void launch_occupancy_bands(const uint32_t *valid, const uint32_t *planes, PlaneGeom g, int64_t t0, int64_t n, int rings, int tp,
                                   uint32_t *occ, cudaStream_t s)
{
    const size_t smem = (size_t) (tp * 8 + 2 * kBandPad + tp) * sizeof(unsigned long long);
    const int vp = occupancy_valid_pitch(g.W);
    for (int64_t i0 = 0; i0 < n; i0 += 65535) {
        const int64_t cnt = n - i0 < 65535 ? n - i0 : 65535;
        occupancy_bands_kernel<<<dim3((unsigned) occupancy_tile_rows(g.H), (unsigned) cnt), kBandThreads, smem, s>>>(
            valid + (size_t) i0 * g.H * CDS_NUM_SECTORS * vp, vp, planes, g, t0 + i0, 2 * rings, tp, occ);
    }
}

void launch_occupancy(const uint32_t *planes, PlaneGeom g, int64_t t0, int64_t n, int rings, int tp,
                      uint32_t *valid_scratch, int64_t scratch_targets, uint32_t *occ, cudaStream_t s, bool valid_ready, bool bands)
{
    if (n == 0) return;
    const int vp = occupancy_valid_pitch(g.W);
    if (valid_ready) {      // the encoder already wrote the bits of targets [0, n) (launch_encode_rgb with `valid`)
        launch_occupancy_kernel(valid_scratch, g.H, vp, tp, t0, n, rings, occ, s);
        if (bands) launch_occupancy_bands(valid_scratch, planes, g, t0, n, rings, tp, occ, s);
        return;
    }
    if (scratch_targets > 32768) scratch_targets = 32768;      // gridDim.y
    for (int64_t i0 = 0; i0 < n; i0 += scratch_targets) {
        const int64_t cnt = n - i0 < scratch_targets ? n - i0 : scratch_targets;
        dim3 grid(g.H, (unsigned) cnt);
        valid_bits_kernel<<<grid, 256, (size_t) CDS_NUM_SECTORS * vp * 4, s>>>(planes, g, t0 + i0, vp, valid_scratch);
        launch_occupancy_kernel(valid_scratch, g.H, vp, tp, t0 + i0, cnt, rings, occ, s);
        if (bands) launch_occupancy_bands(valid_scratch, planes, g, t0 + i0, cnt, rings, tp, occ, s);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Mask preparation: ordered compaction of the pixels above the mask threshold and outside the label regions.
// Pass 1 counts per (mask, row); pass 2 turns counts into row starts; pass 3 writes the records.  One warp per row.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool in_rects(const RectSet &r, int x, int y)
{
    bool in = false;
#pragma unroll
    for (int i = 0; i < 8; i++)
        if (i < r.n) in |= (x >= r.x0[i] && x < r.x1[i] && y >= r.y0[i] && y < r.y1[i]);
    return in;
}

__global__ void __launch_bounds__(128) mask_count_rows_kernel(const uint8_t *__restrict__ rgb, int W, int H, int thr, RectSet rects,
                                                              uint32_t *__restrict__ rowcount)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int y = blockIdx.x * 4 + warp;
    const int m = blockIdx.y;
    if (y >= H) return;
    const uint8_t *row = rgb + ((size_t) m * H + y) * W * 3;
    int cnt = 0;
    for (int x = lane; x < W; x += 32) {
        int r = row[3 * x], g = row[3 * x + 1], b = row[3 * x + 2];
        bool pass = (r > thr || g > thr || b > thr) && !in_rects(rects, x, y);
        cnt += pass ? 1 : 0;
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) rowcount[(size_t) m * (H + 1) + y] = (uint32_t) cnt;
}

void launch_mask_count_rows(const uint8_t *rgb, int n_masks, int W, int H, int threshold, RectSet rects,
                            uint32_t *rowcount, cudaStream_t s)
{
    if (n_masks == 0) return;
    dim3 grid((H + 3) / 4, n_masks);
    mask_count_rows_kernel<<<grid, 128, 0, s>>>(rgb, W, H, threshold, rects, rowcount);
}

// in place: rowcount[m][0..H) counts  ->  rowcount[m][0..H] exclusive starts (last = P)
__global__ void mask_scan_rows_kernel(uint32_t *__restrict__ rowcount, int n_masks, int H, int32_t *__restrict__ sizes)
{
    int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_masks) return;
    uint32_t *rc = rowcount + (size_t) m * (H + 1);
    uint32_t acc = 0;
    for (int y = 0; y < H; y++) { uint32_t c = rc[y]; rc[y] = acc; acc += c; }
    rc[H] = acc;
    sizes[m] = (int32_t) acc;
}

void launch_mask_scan_rows(uint32_t *rowcount, int n_masks, int H, int32_t *sizes, cudaStream_t s)
{
    if (n_masks == 0) return;
    mask_scan_rows_kernel<<<(n_masks + 63) / 64, 64, 0, s>>>(rowcount, n_masks, H, sizes);
}

__global__ void __launch_bounds__(128) mask_write_records_kernel(const uint8_t *__restrict__ rgb, int W, int H, int thr, RectSet rects,
                                                                 const uint32_t *__restrict__ rowstart, const uint64_t *__restrict__ rec_offset,
                                                                 const uint16_t *__restrict__ rank_tab,
                                                                 const cds_class_interval *__restrict__ class_tab,
                                                                 cds_mask_record *__restrict__ records, uint32_t *__restrict__ classes)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int y = blockIdx.x * 4 + warp;
    const int m = blockIdx.y;
    if (y >= H) return;
    const uint8_t *row = rgb + ((size_t) m * H + y) * W * 3;
    cds_mask_record *out = records + rec_offset[m] + rowstart[(size_t) m * (H + 1) + y];
    uint32_t *cls_out = classes + rec_offset[m] + rowstart[(size_t) m * (H + 1) + y];
    int run = 0;
    for (int x0 = 0; x0 < W; x0 += 32) {
        int x = x0 + lane;
        bool pass = false;
        int r = 0, g = 0, b = 0;
        if (x < W) {
            r = row[3 * x]; g = row[3 * x + 1]; b = row[3 * x + 2];
            pass = (r > thr || g > thr || b > thr) && !in_rects(rects, x, y);
        }
        unsigned bal = __ballot_sync(0xffffffffu, pass);
        if (pass) {
            int second, maxv;
            int sector = classify_color_dev(r, g, b, second, maxv);
            cds_mask_record rec;
            rec.xy = (uint32_t) x | ((uint32_t) y << 16);
            rec.lo1 = CDS_EMPTY_LO; rec.lo2 = CDS_EMPTY_LO; rec.lens = 0;
            uint32_t cls = CDS_CLASS_NONE_INDEX;
            if (sector >= 0) {
                int rank = __ldg(rank_tab + second * 256 + maxv);
                cls = (uint32_t) (sector * CDS_NUM_RANKS + rank);
                cds_class_interval iv = class_tab[sector * CDS_NUM_RANKS + rank];
                uint32_t len1 = 0, len2 = 0;
                if (iv.lo1 != CDS_IV_EMPTY) { rec.lo1 = iv.lo1 << CDS_CODE_SR_SHIFT; len1 = iv.len1; }
                if (iv.lo2 != CDS_IV_EMPTY) { rec.lo2 = iv.lo2 << CDS_CODE_SR_SHIFT; len2 = iv.len2; }
                rec.lens = len1 | (len2 << 16);
            }
            int idx = run + __popc(bal & ((1u << lane) - 1));
            out[idx] = rec;
            cls_out[idx] = cls;
        }
        run += __popc(bal);
    }
}

void launch_mask_write_records(const uint8_t *rgb, int n_masks, int W, int H, int threshold, RectSet rects,
                               const uint32_t *rowstart, const uint64_t *rec_offset, const uint16_t *rank_tab,
                               const cds_class_interval *class_tab, cds_mask_record *records, uint32_t *classes, cudaStream_t s)
{
    if (n_masks == 0) return;
    dim3 grid((H + 3) / 4, n_masks);
    mask_write_records_kernel<<<grid, 128, 0, s>>>(rgb, W, H, threshold, rects, rowstart, rec_offset, rank_tab, class_tab, records, classes);
}

// ------------------------------------------------------------------------------------------------------------------
// Palettes of the compact mask records (cds_common.h): per group of CDS_PALETTE_GROUP masks, mark the colour classes in
// use, number them, pack their intervals, rewrite the records as x | y << 11 | index << 21.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kClassSlots = CDS_NUM_CLASSES + 1;

__global__ void __launch_bounds__(256) palette_mark_kernel(const MaskClassRef *__restrict__ masks, uint32_t *__restrict__ flags)
{
    const int m = blockIdx.y;
    const MaskClassRef mr = masks[m];
    uint32_t *f = flags + (size_t) (m / CDS_PALETTE_GROUP) * kClassSlots;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < mr.P; i += gridDim.x * blockDim.x) f[mr.classes[i]] = 1u;
}

void launch_palette_mark(const MaskClassRef *masks, int n_masks, uint32_t *flags, cudaStream_t s)
{
    for (int m0 = 0; m0 < n_masks; m0 += 32768) {      // multiple of CDS_PALETTE_GROUP, so group numbering stays aligned
        int cnt = n_masks - m0 < 32768 ? n_masks - m0 : 32768;
        dim3 grid(8, cnt);
        palette_mark_kernel<<<grid, 256, 0, s>>>(masks + m0, flags + (size_t) (m0 / CDS_PALETTE_GROUP) * kClassSlots);
    }
}

__global__ void __launch_bounds__(1024) palette_scan_kernel(const uint32_t *__restrict__ flags, uint32_t *__restrict__ pidx,
                                                            int32_t *__restrict__ n_pal)
{
    __shared__ uint32_t s_part[1024];
    const int g = blockIdx.x;
    const uint32_t *f = flags + (size_t) g * kClassSlots;
    uint32_t *o = pidx + (size_t) g * kClassSlots;
    const int per = (kClassSlots + 1023) / 1024;
    const int lo = threadIdx.x * per, hi = min(lo + per, kClassSlots);
    uint32_t sum = 0;
    for (int i = lo; i < hi; i++) sum += f[i];
    s_part[threadIdx.x] = sum;
    __syncthreads();
    // Hillis-Steele inclusive scan over the 1024 partial sums
    for (int off = 1; off < 1024; off <<= 1) {
        uint32_t v = threadIdx.x >= off ? s_part[threadIdx.x - off] : 0u;
        __syncthreads();
        s_part[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t acc = s_part[threadIdx.x] - sum;
    for (int i = lo; i < hi; i++) { o[i] = acc; acc += f[i]; }
    if (threadIdx.x == 1023) n_pal[g] = (int32_t) s_part[1023];
}

void launch_palette_scan(const uint32_t *flags, int n_groups, uint32_t *pidx, int32_t *n_pal, cudaStream_t s)
{
    if (n_groups == 0) return;
    palette_scan_kernel<<<n_groups, 1024, 0, s>>>(flags, pidx, n_pal);
}

__device__ __forceinline__ uint32_t pack_palette_word(uint32_t lo, uint32_t len)
{
    if (lo == CDS_IV_EMPTY || len > CDS_PAL_MAX_LEN) return CDS_PAL_EMPTY_LO;   // callers never build palettes when a length overflows
    return lo | (len << CDS_PAL_LO_BITS);
}

__global__ void __launch_bounds__(256) palette_fill_kernel(const uint32_t *__restrict__ flags, const uint32_t *__restrict__ pidx,
                                                           const cds_class_interval *__restrict__ class_tab, uint2 *__restrict__ palettes)
{
    const int g = blockIdx.y;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= kClassSlots) return;
    if (!flags[(size_t) g * kClassSlots + c]) return;
    const uint32_t idx = pidx[(size_t) g * kClassSlots + c];
    if (idx >= CDS_PALETTE_SIZE) return;
    uint2 e = make_uint2(CDS_PAL_EMPTY_LO, CDS_PAL_EMPTY_LO);
    if (c < CDS_NUM_CLASSES) {
        const cds_class_interval iv = class_tab[c];
        e.x = pack_palette_word(iv.lo1, iv.len1);
        e.y = pack_palette_word(iv.lo2, iv.len2);
    }
    palettes[(size_t) g * CDS_PALETTE_SIZE + idx] = e;
}

void launch_palette_fill(const uint32_t *flags, const uint32_t *pidx, int n_groups, const cds_class_interval *class_tab,
                         uint2 *palettes, cudaStream_t s)
{
    for (int g0 = 0; g0 < n_groups; g0 += 32768) {
        int cnt = n_groups - g0 < 32768 ? n_groups - g0 : 32768;
        dim3 grid((kClassSlots + 255) / 256, cnt);
        palette_fill_kernel<<<grid, 256, 0, s>>>(flags + (size_t) g0 * kClassSlots, pidx + (size_t) g0 * kClassSlots, class_tab,
                                                 palettes + (size_t) g0 * CDS_PALETTE_SIZE);
    }
}

__global__ void __launch_bounds__(256) palette_records_kernel(const MaskClassRef *__restrict__ masks, const uint32_t *__restrict__ pidx,
                                                              const int32_t *__restrict__ n_pal)
{
    const int m = blockIdx.y;
    const int g = m / CDS_PALETTE_GROUP;
    if (n_pal[g] >= CDS_PALETTE_SIZE) return;   // the last index is reserved for idle lanes
    const MaskClassRef mr = masks[m];
    const uint32_t *px = pidx + (size_t) g * kClassSlots;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < mr.P; i += gridDim.x * blockDim.x) {
        const uint32_t xy = mr.records[i].xy;
        mr.crec[i] = (xy & 0x7FFu) | (((xy >> 16) & 0x3FFu) << 11) | (px[mr.classes[i]] << 21);
    }
}

void launch_palette_records(const MaskClassRef *masks, int n_masks, const uint32_t *pidx, const int32_t *n_pal, cudaStream_t s)
{
    for (int m0 = 0; m0 < n_masks; m0 += 32768) {
        int cnt = n_masks - m0 < 32768 ? n_masks - m0 : 32768;
        dim3 grid(8, cnt);
        palette_records_kernel<<<grid, 256, 0, s>>>(masks + m0, pidx + (size_t) (m0 / CDS_PALETTE_GROUP) * kClassSlots,
                                                    n_pal + m0 / CDS_PALETTE_GROUP);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Generic pixel match: one CTA per (target, mask); gathers straight from the HBM/L2-resident code plane with explicit
// bounds checks, so any even xyShift works.  Used when the band kernel does not apply (few masks, xyShift > 4) and as
// the simple second implementation the band kernel is cross-checked against.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool code_matches(uint32_t c, uint32_t lo1, uint32_t len1, uint32_t lo2, uint32_t len2)
{
    return (c - lo1 <= len1) | (c - lo2 <= len2);
}

__global__ void __launch_bounds__(256) pixelmatch_gather_kernel(const MaskDesc *__restrict__ masks, const uint32_t *__restrict__ planes,
                                                                PlaneGeom g, int64_t n_targets, ShiftSet shifts,
                                                                int32_t *__restrict__ scores)
{
    __shared__ int warp_sums[8];
    __shared__ int s_total;
    const int64_t t = blockIdx.x;
    const int m = blockIdx.y;
    const MaskDesc md = masks[m];
    const uint32_t *plane = planes + g.row_offset(t, 0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int best[2] = {0, 0};
    const int n_orient = shifts.mirror ? 2 : 1;
    for (int o = 0; o < n_orient; o++) {
        for (int v = 0; v < shifts.n; v++) {
            const int dx = shifts.dx[v], dy = shifts.dy[v];
            int cnt = 0;
            for (int i = threadIdx.x; i < md.P; i += blockDim.x) {
                const uint4 q = __ldg(reinterpret_cast<const uint4 *>(md.records + i));
                int x = (int) (q.x & 0xFFFFu) + dx;
                int y = (int) (q.x >> 16) + dy;
                if (x >= 0 && x < g.W && y >= 0 && y < g.H) {          // shiftMaskPosArray :138-141
                    if (o) x = g.W - 1 - x;                             // mirrorMask :153-154 (applied after the shift)
                    uint32_t c = __ldg(plane + (size_t) y * g.pitch + x);
                    uint32_t len1 = ((q.w & 0xFFFFu) << CDS_CODE_SR_SHIFT) | 0xFFu;
                    uint32_t len2 = ((q.w >> 16) << CDS_CODE_SR_SHIFT) | 0xFFu;
                    cnt += code_matches(c, q.y, len1, q.z, len2) ? 1 : 0;
                }
            }
            cnt = __reduce_add_sync(0xffffffffu, cnt);
            if (lane == 0) warp_sums[warp] = cnt;
            __syncthreads();
            if (threadIdx.x == 0) {
                int tot = 0;
                for (int w = 0; w < (int) (blockDim.x >> 5); w++) tot += warp_sums[w];
                s_total = tot;
            }
            __syncthreads();
            best[o] = max(best[o], s_total);
        }
    }
    if (threadIdx.x == 0) {
        int score = best[0];
        int mir = 0;
        if (shifts.mirror && best[1] > best[0]) { score = best[1]; mir = 1; }   // strict :189
        scores[(size_t) m * n_targets + t] = score | (mir ? CDS_SCORE_MIRROR_BIT : 0);
    }
}

void launch_pixelmatch_gather(const MaskDesc *masks, int n_masks, const uint32_t *planes, PlaneGeom g,
                              int64_t n_targets, ShiftSet shifts, int32_t *scores, cudaStream_t s)
{
    if (n_masks == 0 || n_targets == 0) return;
    // gridDim.y <= 65535
    for (int m0 = 0; m0 < n_masks; m0 += 32768) {
        int cnt = n_masks - m0 < 32768 ? n_masks - m0 : 32768;
        dim3 grid((unsigned) n_targets, (unsigned) cnt);
        pixelmatch_gather_kernel<<<grid, 256, 0, s>>>(masks + m0, planes, g, n_targets, shifts, scores + (size_t) m0 * n_targets);
    }
}

}  // namespace cds

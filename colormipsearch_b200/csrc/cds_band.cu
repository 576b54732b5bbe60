// cds_band.cu -- batched pixel match: target row bands staged in shared memory by TMA bulk copies, a group of masks
// streamed against each band, match counts kept as packed 16-bit lanes in registers.
//
// What it computes is exactly PixelMatchColorDepthSearchAlgorithm.calculateMatchingScore
// (colormipsearch-api/src/main/java/org/janelia/colormipsearch/cds/PixelMatchColorDepthSearchAlgorithm.java:166-263) for every
// (mask, target) of the launch: per shift/mirror variant the number of mask pixels whose shifted target pixel is inside the
// image, above the data threshold and within zTolerance on the colour-depth scale; max over the unmirrored variants, max over
// the mirrored ones, mirrored wins only when strictly greater.
//
// How (B200):
//   * work item = (mask group of GROUP masks, target).  Items are ordered group-major so that all CTAs stream the SAME
//     group's pixel records (L2-resident) while each target plane is read from HBM once per group.
//   * a persistent grid of one CTA per SM: NCW consumer warps + 1 producer warp.  The target is consumed as bands of R rows
//     (+ s = xyShift halo rows on both sides).  A band of a plane is ONE contiguous span of HBM (cds_kernels.cuh PlaneGeom),
//     fetched by a single cp.async.bulk (TMA bulk copy, SASS UBLKCP) that completes on a "full" mbarrier.  Two stages; the
//     producer refills a stage as soon as every consumer warp has arrived on its "empty" mbarrier, so there is no CTA-wide
//     barrier per band and warps may run one band ahead of stragglers.  The producer also pulls the work items from a
//     global counter and publishes them to the consumers through shared memory.
//   * out-of-image pixels of shifted / mirrored variants need no bounds test: they land in the pad columns / guard rows of
//     the plane (or the pad words placed below each stage), whose code words can never match.
//   * next to every band the producer also fetches the matching rows of the library's occupancy bitmap (one bit per pixel:
//     "some shifted position of this pixel is above the data threshold").  A warp skips the 9 (17) evaluations of an
//     orientation when none of its 32 mask pixels has its bit set -- exact, because a clear bit means every shifted target
//     pixel is below the threshold.  Colour-depth MIPs are ~95 % black, so most warp iterations are skipped.
//   * inside a band, consumer warps grab tickets = (mask, chunk of CHUNK records of that mask inside the band) from a shared
//     counter; a lane owns one mask pixel per iteration: one LDG.128 for the record (prefetched one iteration ahead), one
//     LDS per variant, two subtract/compare pairs and one predicated add into a packed counter.  A ticket ends with one
//     REDUX per packed register and shared-memory atomic adds into the per-(mask, variant) accumulators.
#include "cds_band.cuh"
#include "cds_ptx.cuh"

#include <cstdlib>

namespace cds {

namespace {

constexpr int kStages = 2;
constexpr int kMaxBands = 128;
constexpr int kPrePad = 4;          // words (16 bytes, keeps the bulk-copy destination aligned)
constexpr int kChunk = 256;         // records per ticket

struct BandParams {
    const MaskDesc *masks;
    int n_masks;
    const uint32_t *planes;
    PlaneGeom g;
    int64_t n_targets;
    int32_t *scores;                // [n_masks][n_targets]
    unsigned long long *work_counter;
    int rows_per_band;              // R
    int n_bands;
    int stage_words;                // (R + 2s) * pitch
    int n_groups;
    const uint32_t *occ;            // occupancy bitmaps in 8 x 4 tiles (cds_kernels.cuh); this kernel uses the all-sector row
    int bpitch;
    const PaletteGroup *groups;     // palette group of masks[0] onwards (masks[0] is CDS_PALETTE_GROUP aligned in the mask set)
};

// cnt += INC when the code word c lies in [lo1, lo1+len1] or [lo2, lo2+len2]: two subtracts, two compares, one predicated add
template <uint32_t INC>
__device__ __forceinline__ void count_hit(uint32_t &cnt, uint32_t c, uint32_t lo1, uint32_t len1, uint32_t lo2, uint32_t len2)
{
    asm("{\n\t.reg .pred p;\n\t.reg .u32 a, b;\n\t"
        "sub.u32 a, %1, %2;\n\t"
        "sub.u32 b, %1, %4;\n\t"
        "setp.le.u32 p, a, %3;\n\t"
        "setp.le.or.u32 p, b, %5, p;\n\t"
        "@p add.u32 %0, %0, %6;\n\t}"
        : "+r"(cnt) : "r"(c), "r"(lo1), "r"(len1), "r"(lo2), "r"(len2), "n"(INC));
}

// shift offsets of ring structure NRINGS (0: none, 1: +-2, 2: +-2 and +-4)
template <int NRINGS> struct Offsets;
template <> struct Offsets<0> { static constexpr int N = 1; };
template <> struct Offsets<1> { static constexpr int N = 9; };
template <> struct Offsets<2> { static constexpr int N = 17; };

template <int NRINGS>
__device__ __forceinline__ void offset_of(int v, int &dx, int &dy)
{
    // v is a compile-time constant after unrolling
    if (NRINGS == 0) { dx = 0; dy = 0; return; }
    if (v < 9) { dx = (v / 3 - 1) * 2; dy = (v % 3 - 1) * 2; return; }
    // ring 4 without its centre: xx in {-4,0,4} x yy in {-4,0,4} minus (0,0)
    int k = v - 9;
    if (k >= 4) k++;
    dx = (k / 3 - 1) * 4;
    dy = (k % 3 - 1) * 4;
}

// The evaluations of one mask pixel against the band in shared memory: NS shifted reads around the pixel (if any lane of
// the warp can match there) and NS around its mirror image.
template <int NRINGS, bool MIRROR, int NREG>
__device__ __forceinline__ void eval_pixel(const uint32_t *__restrict__ rowbase, int pitch, int x, int xm, bool any_n, bool any_m,
                                           uint32_t lo1, uint32_t len1, uint32_t lo2, uint32_t len2, uint32_t (&cnt)[NREG])
{
    constexpr int NS = Offsets<NRINGS>::N;
    if (any_n) {
        const uint32_t *pc = rowbase + x;                                    // unmirrored centre
#pragma unroll
        for (int v = 0; v < NS; v++) {
            int dx, dy;
            offset_of<NRINGS>(v, dx, dy);
            const uint32_t c = pc[dy * pitch + dx];
            if (v & 1) count_hit<0x10000u>(cnt[v >> 1], c, lo1, len1, lo2, len2);
            else count_hit<1u>(cnt[v >> 1], c, lo1, len1, lo2, len2);
        }
    }
    if (MIRROR && any_m) {
        const uint32_t *pm = rowbase + xm;                                   // mirrored centre
#pragma unroll
        for (int v = 0; v < NS; v++) {
            int dx, dy;
            offset_of<NRINGS>(v, dx, dy);
            const uint32_t c = pm[dy * pitch - dx];                          // mirror of (x + dx) is (W-1-x) - dx
            if ((NS + v) & 1) count_hit<0x10000u>(cnt[(NS + v) >> 1], c, lo1, len1, lo2, len2);
            else count_hit<1u>(cnt[(NS + v) >> 1], c, lo1, len1, lo2, len2);
        }
    }
}

// Shared-memory layout, identical on host (sizing) and device (carving).
template <int GROUP>
struct BandSmem {
    size_t stage_off, bits_off, pal_off, acc_off, seg_off, tick_off, rec_off, bar_off, next_off, item_off, total;
    __host__ __device__ BandSmem(int stage_words, int n_bands, int NV, int bits_words)
    {
        size_t o = 0;
        stage_off = o; o += (size_t) kStages * (stage_words + kPrePad) * 4;
        bits_off = o;  o += (size_t) kStages * bits_words * 4;
        pal_off = o;   o += (size_t) CDS_PALETTE_SIZE * 8;
        acc_off = o;   o += (size_t) GROUP * NV * 4;
        seg_off = o;   o += (size_t) GROUP * (n_bands + 1) * 4;
        tick_off = o;  o += ((size_t) n_bands * (GROUP + 1) * 2 + 15) / 16 * 16;
        rec_off = o;   o += (size_t) GROUP * 8;
        bar_off = o;   o += 2 * kStages * 8;
        next_off = o;  o += 16;
        item_off = o;  o += 16;
        total = o;
    }
};

template <int NRINGS, bool MIRROR, int GROUP, int NCW>
__global__ void __launch_bounds__((NCW + 1) * 32, 1) pixelmatch_band_kernel(const BandParams p)
{
    constexpr int NS = Offsets<NRINGS>::N;            // variants per orientation
    constexpr int NV = MIRROR ? 2 * NS : NS;          // variants
    constexpr int NREG = (NV + 1) / 2;                // packed 16-bit counter registers
    constexpr int S = 2 * NRINGS;                     // halo rows = xyShift
    constexpr int NCT = NCW * 32;                     // consumer threads

    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int rowpitch = occupancy_row_pitch(p.bpitch);
    const int any_off = occupancy_any_offset(p.bpitch);      // the OR over the sectors
    const int bits_words = (p.rows_per_band / 4) * rowpitch;       // rows_per_band is a multiple of the tile height
    const BandSmem<GROUP> L(p.stage_words, p.n_bands, NV, bits_words);
    uint32_t *s_stage = reinterpret_cast<uint32_t *>(smem_raw + L.stage_off) + kPrePad;
    const int stage_stride = p.stage_words + kPrePad;
    const uint32_t *s_bits = reinterpret_cast<const uint32_t *>(smem_raw + L.bits_off);  // [kStages][R * bpitch]
    uint2 *s_pal = reinterpret_cast<uint2 *>(smem_raw + L.pal_off);                      // palette of the current group
    int *s_acc = reinterpret_cast<int *>(smem_raw + L.acc_off);                         // [GROUP][NV]
    uint32_t *s_seg = reinterpret_cast<uint32_t *>(smem_raw + L.seg_off);               // [GROUP][n_bands + 1] record index at band starts
    uint16_t *s_tick = reinterpret_cast<uint16_t *>(smem_raw + L.tick_off);             // [n_bands][GROUP + 1] ticket prefix sums
    const void **s_rec = reinterpret_cast<const void **>(smem_raw + L.rec_off);         // record arrays (compact or 16-byte)
    unsigned long long *s_full = reinterpret_cast<unsigned long long *>(smem_raw + L.bar_off);
    unsigned long long *s_empty = s_full + kStages;
    int *s_next = reinterpret_cast<int *>(smem_raw + L.next_off);                       // [kStages] ticket counters
    long long *s_item = reinterpret_cast<long long *>(smem_raw + L.item_off);           // [2] published work items

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int pitch = p.g.pitch, W = p.g.W, H = p.g.H, R = p.rows_per_band, NB = p.n_bands;
    const long long n_items = (long long) p.n_groups * p.n_targets;

    if (tid == 0) {
        for (int s = 0; s < kStages; s++) {
            mbar_init(smem_u32(s_full + s), 1);
            mbar_init(smem_u32(s_empty + s), NCW);
            s_next[s] = 0;
        }
        mbar_fence_init();
    }
    for (int i = tid; i < GROUP * NV; i += blockDim.x) s_acc[i] = 0;
    // never-matching words below each stage: a pixel in the first row of a band whose shifted / mirrored column is -1..-4
    if (tid < kStages * kPrePad) s_stage[(tid / kPrePad) * stage_stride - kPrePad + (tid % kPrePad)] = CDS_CODE_PAD_WORD;
    __syncthreads();

    if (warp == NCW) {
        // ------------------------------------------------------------------ producer (one lane)
        if (lane == 0) {
            uint32_t q = 0;                 // running band number across items: stage = q & 1, use = q >> 1
            uint32_t iseq = 0;
            for (;;) {
                const long long w = (long long) atomicAdd(p.work_counter, 1ull);
                const bool done = w >= n_items;
                const int nb = done ? 1 : NB;
                for (int b = 0; b < nb; b++, q++) {
                    const int stage = q & 1;
                    if (q >= kStages) mbar_wait(smem_u32(s_empty + stage), ((q >> 1) - 1) & 1);
                    s_next[stage] = 0;
                    if (b == 0) s_item[iseq & 1] = done ? -1 : w;
                    const uint32_t bar = smem_u32(s_full + stage);
                    if (done) { mbar_arrive(bar); break; }
                    const int64_t t = w % p.n_targets;
                    const int y0 = b * R;
                    const int y1 = min(y0 + R, H);
                    const uint32_t bytes = (uint32_t) ((y1 - y0 + 2 * S) * pitch) * 4u;
                    const uint32_t *src = p.planes + p.g.row_offset(t, 0) + (long long) (y0 - S) * pitch;   // guard rows cover y0 - S < 0
                    const uint32_t bbytes = (uint32_t) (((y1 - y0 + 3) / 4) * rowpitch) * 4u;
                    const uint32_t *bsrc = p.occ + ((size_t) t * occupancy_tile_rows(H) + y0 / 4) * rowpitch;
                    mbar_expect_tx(bar, bytes + bbytes);
                    bulk_load(smem_u32(s_stage + (size_t) stage * stage_stride), src, bytes, bar);
                    bulk_load(smem_u32(s_bits + (size_t) stage * bits_words), bsrc, bbytes, bar);
                }
                if (done) break;
                iseq++;
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumers
    uint32_t q = 0, iseq = 0;
    int cur_gi = -1;
    bool compact = false;
    for (;;) {
        mbar_wait(smem_u32(s_full + (q & 1)), (q >> 1) & 1);
        const long long w = *reinterpret_cast<volatile long long *>(s_item + (iseq & 1));
        if (w < 0) break;
        const int gi = (int) (w / p.n_targets);
        const int64_t t = w % p.n_targets;
        const int m0 = gi * GROUP;
        const int mb = min(GROUP, p.n_masks - m0);

        if (gi != cur_gi) {
            // per-group tables: record base pointers, band boundaries and per-band ticket prefix sums.  Every consumer passed
            // the barrier that ends the previous item, so nobody still reads the old tables.
            const PaletteGroup pg = p.groups[m0 / CDS_PALETTE_GROUP];
            compact = pg.palette != nullptr;
            for (int i = tid; i < mb; i += NCT)
                s_rec[i] = compact ? (const void *) p.masks[m0 + i].crec : (const void *) p.masks[m0 + i].records;
            if (compact) {
                for (int i = tid; i < pg.n_pal; i += NCT) s_pal[i] = pg.palette[i];
                if (tid == 0) s_pal[CDS_PALETTE_SIZE - 1] = make_uint2(CDS_PAL_EMPTY_LO, CDS_PAL_EMPTY_LO);   // idle lanes point here
            }
            for (int i = tid; i < mb * (NB + 1); i += NCT) {
                const int mi = i / (NB + 1), b = i % (NB + 1);
                s_seg[i] = __ldg(p.masks[m0 + mi].rowstart + min(b * R, H));
            }
            consumer_barrier<NCT>();
            for (int b = tid; b < NB; b += NCT) {
                uint32_t acc = 0;
                uint16_t *row = s_tick + b * (GROUP + 1);
                for (int mi = 0; mi < GROUP; mi++) {
                    row[mi] = (uint16_t) acc;
                    if (mi < mb) acc += (s_seg[mi * (NB + 1) + b + 1] - s_seg[mi * (NB + 1) + b] + kChunk - 1) / kChunk;
                }
                row[GROUP] = (uint16_t) acc;
            }
            consumer_barrier<NCT>();
            cur_gi = gi;
        }

        for (int b = 0; b < NB; b++, q++) {
            const int stage = q & 1;
            if (b > 0) mbar_wait(smem_u32(s_full + stage), (q >> 1) & 1);
            const uint32_t *band = s_stage + (size_t) stage * stage_stride;
            const int y0 = b * R;
            const uint16_t *tick = s_tick + b * (GROUP + 1);
            const int n_tickets = tick[GROUP];

            for (;;) {
                int tk = 0;
                if (lane == 0) tk = atomicAdd(&s_next[stage], 1);
                tk = __shfl_sync(0xffffffffu, tk, 0);
                if (tk >= n_tickets) break;
                // mask of the ticket: the last mi with tick[mi] <= tk
                int le = 0;
#pragma unroll
                for (int k = 0; k < GROUP / 32; k++) le += __popc(__ballot_sync(0xffffffffu, (int) tick[k * 32 + lane] <= tk));
                const int mi = le - 1;
                const uint32_t seg_end = s_seg[mi * (NB + 1) + b + 1];
                const uint32_t seg0 = s_seg[mi * (NB + 1) + b] + (uint32_t) (tk - tick[mi]) * kChunk;
                const uint32_t seg1 = min(seg0 + kChunk, seg_end);
                uint32_t cnt[NREG];
#pragma unroll
                for (int j = 0; j < NREG; j++) cnt[j] = 0;
                const uint32_t *bits = s_bits + (size_t) stage * bits_words;

                // every lane runs the same number of iterations (the occupancy votes are warp-wide); lanes past the end of
                // the chunk carry a record that cannot match and sits on a valid address
                if (compact) {
                    const uint32_t *cr = static_cast<const uint32_t *>(s_rec[mi]);
                    const uint32_t idle = ((uint32_t) y0 << 11) | ((uint32_t) (CDS_PALETTE_SIZE - 1) << 21);
                    // records are prefetched four iterations ahead
                    uint32_t r0 = idle, r1 = idle, r2 = idle, r3 = idle;
                    if (seg0 + lane < seg1) r0 = __ldg(cr + seg0 + lane);
                    if (seg0 + 32 + lane < seg1) r1 = __ldg(cr + seg0 + 32 + lane);
                    if (seg0 + 64 + lane < seg1) r2 = __ldg(cr + seg0 + 64 + lane);
                    if (seg0 + 96 + lane < seg1) r3 = __ldg(cr + seg0 + 96 + lane);
                    for (uint32_t base = seg0; base < seg1; base += 32) {
                        const uint32_t cur = r0;
                        r0 = r1; r1 = r2; r2 = r3;
                        const uint32_t inext = base + 128 + lane;
                        r3 = idle;
                        if (inext < seg1) r3 = __ldg(cr + inext);
                        const int x = (int) (cur & 0x7FFu);
                        const int brow = (int) ((cur >> 11) & 0x3FFu) - y0;
                        const int xm = W - 1 - x;
                        const bool live = base + lane < seg1;
                        const uint32_t wn = bits[(brow >> 2) * rowpitch + any_off + (x >> 3)];
                        const uint32_t wm = bits[(brow >> 2) * rowpitch + any_off + (xm >> 3)];
                        const bool any_n = __any_sync(0xffffffffu, live && ((wn >> ((brow & 3) * 8 + (x & 7))) & 1u));
                        const bool any_m = MIRROR && __any_sync(0xffffffffu, live && ((wm >> ((brow & 3) * 8 + (xm & 7))) & 1u));
                        if (!any_n && !any_m) continue;
                        const uint2 pe = s_pal[cur >> 21];
                        const uint32_t lo1 = (pe.x & ((1u << CDS_PAL_LO_BITS) - 1)) << CDS_CODE_SR_SHIFT;
                        const uint32_t len1 = ((pe.x >> CDS_PAL_LO_BITS) << CDS_CODE_SR_SHIFT) | 0xFFu;
                        const uint32_t lo2 = (pe.y & ((1u << CDS_PAL_LO_BITS) - 1)) << CDS_CODE_SR_SHIFT;
                        const uint32_t len2 = ((pe.y >> CDS_PAL_LO_BITS) << CDS_CODE_SR_SHIFT) | 0xFFu;
                        eval_pixel<NRINGS, MIRROR, NREG>(band + (brow + S) * pitch, pitch, x, xm, any_n, any_m, lo1, len1, lo2, len2, cnt);
                    }
                } else {
                    const cds_mask_record *rec = static_cast<const cds_mask_record *>(s_rec[mi]);
                    const uint4 idle = make_uint4((uint32_t) y0 << 16, CDS_EMPTY_LO, CDS_EMPTY_LO, 0u);
                    uint4 qr = idle;
                    if (seg0 + lane < seg1) qr = __ldg(reinterpret_cast<const uint4 *>(rec + seg0 + lane));
                    for (uint32_t base = seg0; base < seg1; base += 32) {
                        const uint4 cur = qr;
                        const uint32_t inext = base + 32 + lane;
                        qr = idle;
                        if (inext < seg1) qr = __ldg(reinterpret_cast<const uint4 *>(rec + inext));   // prefetch behind the compute
                        const int x = (int) (cur.x & 0xFFFFu);
                        const int brow = (int) (cur.x >> 16) - y0;
                        const int xm = W - 1 - x;
                        const bool live = base + lane < seg1;
                        const uint32_t wn = bits[(brow >> 2) * rowpitch + any_off + (x >> 3)];
                        const uint32_t wm = bits[(brow >> 2) * rowpitch + any_off + (xm >> 3)];
                        const bool any_n = __any_sync(0xffffffffu, live && ((wn >> ((brow & 3) * 8 + (x & 7))) & 1u));
                        const bool any_m = MIRROR && __any_sync(0xffffffffu, live && ((wm >> ((brow & 3) * 8 + (xm & 7))) & 1u));
                        if (!any_n && !any_m) continue;
                        const uint32_t len1 = ((cur.w & 0xFFFFu) << CDS_CODE_SR_SHIFT) | 0xFFu;
                        const uint32_t len2 = ((cur.w >> 16) << CDS_CODE_SR_SHIFT) | 0xFFu;
                        eval_pixel<NRINGS, MIRROR, NREG>(band + (brow + S) * pitch, pitch, x, xm, any_n, any_m, cur.y, len1, cur.z, len2, cnt);
                    }
                }
                // ticket done: warp totals (a ticket has <= kChunk pixels, so the packed halves cannot carry)
                uint32_t mine0 = 0, mine1 = 0;
#pragma unroll
                for (int j = 0; j < NREG; j++) {
                    const uint32_t tot = __reduce_add_sync(0xffffffffu, cnt[j]);
                    if ((lane >> 1) == j) mine0 = tot;
                    if (((lane + 32) >> 1) == j) mine1 = tot;
                }
                const int v0 = (int) ((lane & 1) ? (mine0 >> 16) : (mine0 & 0xFFFFu));
                if (lane < NV && v0) atomicAdd(&s_acc[mi * NV + lane], v0);
                if (NV > 32) {
                    const int v1 = (int) ((lane & 1) ? (mine1 >> 16) : (mine1 & 0xFFFFu));
                    if (lane + 32 < NV && v1) atomicAdd(&s_acc[mi * NV + lane + 32], v1);
                }
            }
            // this warp is done with the stage: let the producer refill it
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(s_empty + stage));
        }

        // item epilogue: max over variants per orientation; mirrored wins only when strictly greater
        consumer_barrier<NCT>();
        for (int mi = tid; mi < mb; mi += NCT) {
            int best = 0, bestm = 0;
#pragma unroll
            for (int v = 0; v < NS; v++) best = max(best, s_acc[mi * NV + v]);
            if (MIRROR) {
#pragma unroll
                for (int v = 0; v < NS; v++) bestm = max(bestm, s_acc[mi * NV + NS + v]);
            }
            int word = best;
            if (MIRROR && bestm > best) word = bestm | CDS_SCORE_MIRROR_BIT;
            p.scores[(size_t) (m0 + mi) * p.n_targets + t] = word;
#pragma unroll
            for (int v = 0; v < NV; v++) s_acc[mi * NV + v] = 0;
        }
        consumer_barrier<NCT>();
        iseq++;
    }
}

struct BandConfig {
    int rows_per_band, n_bands, stage_words;
    size_t smem_bytes;
    bool ok;
};

template <int GROUP>
BandConfig band_config(int xy_shift, bool mirror, const PlaneGeom &g)
{
    const int bpitch = occupancy_tile_pitch(g.W);
    BandConfig c{};
    const int S = xy_shift;
    const int NS = xy_shift == 0 ? 1 : (xy_shift == 2 ? 9 : 17);
    const int NV = mirror ? 2 * NS : NS;
    const size_t budget = 227 * 1024;
    for (int R = (g.H + 3) / 4 * 4; R >= 4; R -= 4) {       // whole occupancy tiles per band
        int n_bands = (g.H + R - 1) / R;
        if (n_bands > kMaxBands) break;
        size_t stage_words = (size_t) (R + 2 * S) * g.pitch;
        if (stage_words * 4 >= (1u << 20)) continue;
        BandSmem<GROUP> L((int) stage_words, n_bands, NV, (R / 4) * occupancy_row_pitch(bpitch));
        if (L.total <= budget) {
            c.rows_per_band = R; c.n_bands = n_bands; c.stage_words = (int) stage_words; c.smem_bytes = L.total; c.ok = true;
            return c;
        }
    }
    c.ok = false;
    return c;
}


int env_int(const char *name, int dflt)
{
    const char *e = std::getenv(name);
    return e ? std::atoi(e) : dflt;
}

template <int GROUP, int NCW>
int launch_cfg(const MaskDesc *masks, int n_masks, const uint32_t *planes, PlaneGeom g, int64_t n_targets,
               const uint32_t *occ, int bpitch, const PaletteGroup *groups, int xy_shift, bool mirror, int32_t *scores,
               const MatchScratch &scratch, cudaStream_t s, int dev)
{
    BandConfig c = band_config<GROUP>(xy_shift, mirror, g);
    if (!c.ok) return 0;
    BandParams p;
    p.masks = masks; p.n_masks = n_masks; p.planes = planes; p.g = g; p.n_targets = n_targets; p.scores = scores;
    p.work_counter = scratch.work_counter;
    p.rows_per_band = c.rows_per_band; p.n_bands = c.n_bands; p.stage_words = c.stage_words;
    p.n_groups = (n_masks + GROUP - 1) / GROUP;
    p.occ = occ; p.bpitch = bpitch; p.groups = groups;
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    long long n_items = (long long) p.n_groups * n_targets;
    int grid = (int) std::min<long long>(n_sm, n_items);
    void (*kern)(const BandParams) = nullptr;
    const int rings = xy_shift / 2;
    if (rings == 0) kern = mirror ? pixelmatch_band_kernel<0, true, GROUP, NCW> : pixelmatch_band_kernel<0, false, GROUP, NCW>;
    else if (rings == 1) kern = mirror ? pixelmatch_band_kernel<1, true, GROUP, NCW> : pixelmatch_band_kernel<1, false, GROUP, NCW>;
    else kern = mirror ? pixelmatch_band_kernel<2, true, GROUP, NCW> : pixelmatch_band_kernel<2, false, GROUP, NCW>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) c.smem_bytes);
    kern<<<grid, (NCW + 1) * 32, c.smem_bytes, s>>>(p);
    return 1;
}

}  // namespace

bool band_kernel_supported(int xy_shift, const PlaneGeom &g)
{
    static const bool disabled = std::getenv("CDSGPU_DISABLE_BAND") != nullptr;
    if (disabled) return false;
    if (!(xy_shift == 0 || xy_shift == 2 || xy_shift == 4)) return false;
    if (xy_shift > g.guard || xy_shift > g.pitch - g.W || xy_shift > kPrePad) return false;
    return band_config<128>(xy_shift, true, g).ok && band_config<64>(xy_shift, true, g).ok;
}

int band_min_masks()
{
    static const int v = env_int("CDSGPU_BAND_MIN_MASKS", 16);
    return v;
}

int launch_pixelmatch_band(const MaskDesc *masks, int n_masks, const uint32_t *planes, PlaneGeom g, int64_t n_targets,
                           const uint32_t *occ, int bpitch, const PaletteGroup *groups, int xy_shift, bool mirror, int32_t *scores,
                           const MatchScratch &scratch, cudaStream_t s)
{
    if (n_masks == 0 || n_targets == 0) return 0;
    if (!occ || !groups || bpitch != occupancy_tile_pitch(g.W)) return 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (!scratch.work_counter) return 0;
    cudaMemsetAsync(scratch.work_counter, 0, sizeof(unsigned long long), s);
    // tuning knobs (defaults picked from profiles/): masks per work item, consumer warps per CTA
    static const int group_env = env_int("CDSGPU_BAND_GROUP", 0);
    static const int warps_env = env_int("CDSGPU_BAND_WARPS", 24);
    const int group = group_env ? group_env : (n_masks > 96 ? 128 : 64);
    if (group == 128) {
        if (warps_env == 24) return launch_cfg<128, 24>(masks, n_masks, planes, g, n_targets, occ, bpitch, groups, xy_shift, mirror, scores, scratch, s, dev);
        return launch_cfg<128, 16>(masks, n_masks, planes, g, n_targets, occ, bpitch, groups, xy_shift, mirror, scores, scratch, s, dev);
    }
    if (warps_env == 24) return launch_cfg<64, 24>(masks, n_masks, planes, g, n_targets, occ, bpitch, groups, xy_shift, mirror, scores, scratch, s, dev);
    return launch_cfg<64, 16>(masks, n_masks, planes, g, n_targets, occ, bpitch, groups, xy_shift, mirror, scores, scratch, s, dev);
}

}  // namespace cds

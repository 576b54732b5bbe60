// cds_cand.cu -- batched pixel match, candidate formulation: 32 mask pixels are tested against a target with ONE AND,
// and only the surviving (pixel, orientation) candidates are evaluated, 32 at a time with every lane busy.
//
// What it computes is exactly PixelMatchColorDepthSearchAlgorithm.calculateMatchingScore
// (colormipsearch-api/src/main/java/org/janelia/colormipsearch/cds/PixelMatchColorDepthSearchAlgorithm.java:166-263) for every
// (mask, target) of the launch, like cds_band.cu (same pipeline, same data, same outputs).  What differs is the inner loop:
//
//   * cds_band.cu gives every lane one mask pixel per iteration and lets a warp skip an orientation when none of its 32
//     pixels has its occupancy bit set.  On colour-depth MIPs ~8 % of the (pixel, orientation) tests can match but ~34 % of
//     the 32-pixel warp iterations contain at least one, so most evaluated lanes are dead weight and the per-pixel
//     bookkeeping (record decode, two bitmap reads, two votes) is paid for every pixel.
//   * here a lane owns one 32-pixel tile WORD of the mask bitmaps per iteration (cds_cand.cuh): candidates = word & occupancy
//     word.  The words of a mask group are ordered by occupancy word, so that tickets of 32 words can be tested against the
//     target ("does it have anything on these tiles, in this sector?") before they are read: ~97 % of them are never scanned.
//     The candidate bits of the words that remain are expanded, load-balanced over the lanes, and evaluated 32 at a time:
//     palette lookup, 9 (17) shifted reads of the band, predicated reductions into per-(mask, variant) counters in global
//     memory.  Work is proportional to the candidates, not to the mask size.
//
// Mirrored variants need no separate code: orientation-1 words are stored in target coordinates (bit W-1-x), and the 3x3
// (5x5) shift pattern is symmetric, so both orientations read the same neighbourhood offsets of their centre; only the
// variant LABEL differs (offset (dx,dy) of a mirrored pixel is the reference's variant (-dx,dy)), and the score is a max
// over labels.  A candidate's orientation just selects the half of the mask's counters it increments.
#include "cds_cand.cuh"
#include "cds_ptx.cuh"

#include <cstdio>
#include <type_traits>
#include <cstdlib>
#include <vector>

namespace cds {

namespace {

constexpr int kMaxStages = 4;     // band stages of the pipeline: CandParams::n_stages of them are used
constexpr int kMaxBands = 256;
constexpr int kPrePad = 4;          // words (16 bytes, keeps the bulk-copy destination aligned)
constexpr int kQueue = 64;          // candidate slots per warp (power of two, >= 2 * 32)
constexpr int kWordQueue = 32;      // word slots per warp: one batch (16 bytes each: candidate bits and what the expansion needs of the entry)
constexpr int kCandOffsetBits = 15; // a staged band has fewer than 2^15 words (227 kB of shared memory hold 2 of them)
constexpr uint32_t kCandOffsetMask = (1u << kCandOffsetBits) - 1u;

struct CandParams {
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
    const uint32_t *occ;            // occupancy bitmaps in 8 x 4 tiles, [n_targets][tile rows][sectors + 1][bpitch] (cds_kernels.cuh)
    int bpitch;
    const PaletteGroup *groups;
    int *acc;                       // [grid][GROUP][2 * offsets] match counters, zero between work items
    int debug_skip;                 // profiling aid (CDSGPU_CAND_NULL): consumers skip the tickets, only the band pipeline runs
    int ticket_skip;                // the lists are in bucket order: a ticket whose occupancy words are all empty is not scanned
    int n_stages;                   // band stages in flight (2 .. kMaxStages)
    int wait_mode;                  // how a warp waits for a band: 0 polls try_wait, 1 try_wait with a suspend-time hint, 2 test_wait + nanosleep
    long long *trace;               // profiling aid (CDSGPU_CAND_TRACE): SM clock of CTA 0's first items, [item][band][32 warps][2] (+ producer in slot 31)
    int band_filter;                // words whose rank-band byte shares no band with the target tile's are dropped (CDSGPU_CAND_NOBAND=1: off)
    int pal_entries;                // palette entries staged in shared memory (cand_staged_palette; 0 for WIDE lists), the last one idle
};
constexpr int kTraceItems = 8;

template <int NRINGS> struct Offsets;
template <> struct Offsets<0> { static constexpr int N = 1; };
template <> struct Offsets<1> { static constexpr int N = 9; };
template <> struct Offsets<2> { static constexpr int N = 17; };

template <int NRINGS>
__device__ __forceinline__ void offset_of(int v, int &dx, int &dy)
{
    if (NRINGS == 0) { dx = 0; dy = 0; return; }
    if (v < 9) { dx = (v / 3 - 1) * 2; dy = (v % 3 - 1) * 2; return; }
    int k = v - 9;                  // ring 4 without its centre
    if (k >= 4) k++;
    dx = (k / 3 - 1) * 4;
    dy = (k % 3 - 1) * 4;
}

// acc[OFF / 4] += 1 (a predicated reduction on this CTA's accumulators in global memory, performed in L2) when the code word c
// lies in [lo, lo + len].  Matches are rare (a few per hundred evaluations), so nearly all of these reductions are predicated
// off; keeping the accumulators out of shared memory leaves room for taller bands.
template <int OFF>
__device__ __forceinline__ void count_hit(const int *acc, uint32_t c, uint32_t lo, uint32_t len)
{
    asm volatile("{\n\t.reg .pred p;\n\t.reg .u32 a;\n\t"
                 "sub.u32 a, %1, %2;\n\t"
                 "setp.le.u32 p, a, %3;\n\t"
                 "@p red.global.add.u32 [%0+%4], 1;\n\t}"
                 :: "l"(acc), "r"(c), "r"(lo), "r"(len), "n"(OFF));
    // no "memory" clobber on purpose: the band reads around it may be scheduled freely; the accumulators are only read after a
    // __threadfence() and a named barrier (a volatile asm with a memory clobber), and volatile asms keep their order
}

// Published by the producer with every stage, so that 31 warps do not each work it out again: the band's part of the group's word list
// and its part of the occupancy rows.
struct __align__(16) BandInfo {
    uint32_t first, end;            // entries [first, end) of the group's word list fall into the band's tile rows
    uint32_t band_lo, band_hi;      // first / last occupancy word index of those tile rows
    uint32_t j_first, n_tk;         // first ticket (of 32 entries) that touches the range, and how many do
    uint32_t n_batches;             // batches of 32 tickets, a multiple of the number of consumer warps
    uint32_t pad;
};

template <int GROUP>
struct CandSmem {
    size_t stage_off, bits_off, pal_off, band_off, queue_off, wqueue_off, bar_off, next_off, item_off, sel_off, total;
    __host__ __device__ CandSmem(int stage_words, int NS, int bits_words, int n_warps, int n_stages, int pal_entries)
    {
        size_t o = 0;
        stage_off = o; o += (size_t) n_stages * (stage_words + kPrePad) * 4;
        bits_off = o;  o += (size_t) n_stages * bits_words * 4;
        pal_off = o;   o += (size_t) pal_entries * 8;                               // a multiple of 16 entries: what follows stays 16-byte aligned
        wqueue_off = o; o += (size_t) n_warps * kWordQueue * 16;
        queue_off = o; o += (size_t) n_warps * kQueue * 8;
        bar_off = o;   o += 2 * kMaxStages * 8;
        item_off = o;  o += 32;                                                 // two published work items {target, group}
        next_off = o;  o += 16;
        o = (o + 15) & ~(size_t) 15;
        band_off = o;  o += (size_t) kMaxStages * 32;                              // per stage: BandInfo
        sel_off = o;   o += 64;                                                 // position of the r-th set bit of a nibble
        (void) NS;
        total = o;
    }
};

// The evaluations of 32 queued candidates: one per lane.
// cand.x = word offset of the candidate's pixel inside the staged band (halo rows included; < 2^15) | (mask inside the group * 2 +
// orientation) << 15 -- everything the evaluation needs as two ready-made offsets, worked out once per WORD by the expansion;
// cand.y = index of the
// candidate's palette reference in the group's lpal array.
template <int NRINGS, int V>
struct EvalUnroll {
    static __device__ __forceinline__ void load(const uint32_t *pc, int pitch, uint32_t (&cw)[Offsets<NRINGS>::N])
    {
        int dx, dy;
        offset_of<NRINGS>(V, dx, dy);
        cw[V] = pc[dy * pitch + dx];
        EvalUnroll<NRINGS, V + 1>::load(pc, pitch, cw);
    }
    static __device__ __forceinline__ void count(const uint32_t (&cw)[Offsets<NRINGS>::N], const int *acc, uint32_t lo, uint32_t len)
    {
        count_hit<4 * V>(acc, cw[V], lo, len);
        EvalUnroll<NRINGS, V + 1>::count(cw, acc, lo, len);
    }
};
template <int NRINGS>
struct EvalUnroll<NRINGS, Offsets<NRINGS>::N> {
    static __device__ __forceinline__ void load(const uint32_t *, int, uint32_t (&)[Offsets<NRINGS>::N]) {}
    static __device__ __forceinline__ void count(const uint32_t (&)[Offsets<NRINGS>::N], const int *, uint32_t, uint32_t) {}
};

// Position of the r-th (0-based) set bit of c, r < popc(c): the byte (= tile row) by three prefix popcounts, the nibble by one
// more, the bit inside the nibble from a 64-byte table (sel[nibble * 4 + r]).  About half the instructions of __fns.
__device__ __forceinline__ uint32_t select_bit(uint32_t c, uint32_t r, const uint8_t *__restrict__ sel)
{
    const uint32_t t0 = (uint32_t) __popc(c & 0xFFu), t1 = (uint32_t) __popc(c & 0xFFFFu), t2 = (uint32_t) __popc(c & 0xFFFFFFu);
    uint32_t sh = 0, e = 0;
    if (r >= t0) { sh = 8; e = t0; }
    if (r >= t1) { sh = 16; e = t1; }
    if (r >= t2) { sh = 24; e = t2; }
    uint32_t b = (c >> sh) & 0xFFu, q = r - e;
    const uint32_t h = (uint32_t) __popc(b & 0xFu);
    if (q >= h) { b >>= 4; q -= h; sh += 4; }
    return sh + sel[(b & 0xFu) * 4 + (q & 3u)];
}

// First half of an evaluation: the candidate's palette reference (palette index | 0x8000 for the second interval), an L2
// access whose latency the caller hides behind the evaluation of the previous batch.  Idle lanes get `idle`, the never-matching entry.
// WIDE (groups with more colour classes than a shared-memory palette holds): lpal carries the packed interval itself, 32 bits per
// set bit, and there is no palette.
template <bool WIDE>
__device__ __forceinline__ uint32_t fetch_palette_ref(uint2 cand, bool live, const uint16_t *__restrict__ lpal, uint64_t policy, uint32_t idle)
{
    if (WIDE) return live ? __ldg(reinterpret_cast<const uint32_t *>(lpal) + cand.y) : CDS_PAL_EMPTY_LO;
    uint32_t pr = idle;
    if (live) pr = policy ? ldg_hint_u16(lpal + cand.y, policy) : (uint32_t) __ldg(lpal + cand.y);
    return pr;
}

template <int NRINGS, bool WIDE>
__device__ __forceinline__ void eval_candidates(uint2 cand, uint32_t pr, const uint32_t *__restrict__ band, int pitch,
                                                const uint2 *__restrict__ s_pal, const int *acc_base)
{
    constexpr int NS = Offsets<NRINGS>::N;
    uint32_t iv = pr;                                                           // WIDE: the reference IS the interval
    if (!WIDE) {
        const uint2 pe = s_pal[pr & 0x7FFFu];                                   // without the "interval 2" flag
        iv = (pr & 0x8000u) ? pe.y : pe.x;                                      // the interval that lives in this candidate's sector
    }
    const uint32_t lo = (iv & ((1u << CDS_PAL_LO_BITS) - 1)) << CDS_CODE_SR_SHIFT;
    const uint32_t len = ((iv >> CDS_PAL_LO_BITS) << CDS_CODE_SR_SHIFT) | 0xFFu;
    const uint32_t *pc = band + (cand.x & (kCandOffsetMask));
    // accumulators of this mask: [0, NS) unmirrored, [NS, 2 NS) mirrored
    const int *acc = acc_base + (cand.x >> kCandOffsetBits);
    (void) NS;
    uint32_t cw[NS];
    EvalUnroll<NRINGS, 0>::load(pc, pitch, cw);          // all shifted reads first, then the compares
    EvalUnroll<NRINGS, 0>::count(cw, acc, lo, len);
}

template <int NRINGS, int GROUP, int NCW, bool HINT, bool WIDE>
__global__ void __launch_bounds__((NCW + 1) * 32, 1) pixelmatch_cand_kernel(const CandParams p)
{
    constexpr int NS = Offsets<NRINGS>::N;            // shift offsets = variants per orientation
    constexpr int NV = 2 * NS;                        // accumulators per mask: [0, NS) unmirrored, [NS, 2NS) mirrored
    constexpr int S = 2 * NRINGS;                     // halo rows = xyShift
    constexpr int NCT = NCW * 32;                     // consumer threads

    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int rowpitch = occupancy_stage_pitch(p.bpitch);          // the staged part of a tile row: sector rows, non-empty bits, band bytes
    const int bits_words = (p.rows_per_band / 4) * rowpitch;       // rows_per_band is a multiple of the tile height
    const int NSTG = p.n_stages;
    const CandSmem<GROUP> L(p.stage_words, NS, bits_words, NCW, NSTG, p.pal_entries);
    uint32_t *s_stage = reinterpret_cast<uint32_t *>(smem_raw + L.stage_off) + kPrePad;
    const int stage_stride = p.stage_words + kPrePad;
    const uint32_t *s_bits = reinterpret_cast<const uint32_t *>(smem_raw + L.bits_off);  // [stages][tile rows of a band * row pitch]
    uint2 *s_pal = reinterpret_cast<uint2 *>(smem_raw + L.pal_off);                      // palette of the current group
    uint2 *s_queue = reinterpret_cast<uint2 *>(smem_raw + L.queue_off);                  // [NCW][kQueue] candidates
    uint4 *s_wqueue = reinterpret_cast<uint4 *>(smem_raw + L.wqueue_off);                // [NCW][kWordQueue] {candidate bits, the word's bits, lrec, meta} of words with candidates
    constexpr int NVP = (NV + 3) / 4 * 4;             // a mask's accumulators padded to whole 16-byte words (the epilogue reads them as int4)
    int *s_acc = p.acc + (size_t) blockIdx.x * GROUP * NVP;                             // this CTA's accumulators [GROUP][NVP], global memory, zero on entry
    BandInfo *s_band = reinterpret_cast<BandInfo *>(smem_raw + L.band_off);             // [kMaxStages] what the consumers need to know about the staged band
    unsigned long long *s_full = reinterpret_cast<unsigned long long *>(smem_raw + L.bar_off);
    unsigned long long *s_empty = s_full + kMaxStages;
    int *s_next = reinterpret_cast<int *>(smem_raw + L.next_off);                       // [stages] batch counters
    long long *s_item = reinterpret_cast<long long *>(smem_raw + L.item_off);           // [2][2] published work items: {target, group}; target -1 = no more work
    uint8_t *s_sel = smem_raw + L.sel_off;                                               // [16][4] r-th set bit of a nibble

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int pitch = p.g.pitch, H = p.g.H, R = p.rows_per_band, NB = p.n_bands;
    const long long n_items = (long long) p.n_groups * p.n_targets;
    const uint64_t pol_stream = HINT ? l2_policy_evict_first() : 0ull, pol_keep = HINT ? l2_policy_evict_last() : 0ull;
    long long *const trace = blockIdx.x == 0 ? p.trace : nullptr;

    if (tid == 0) {
        for (int s = 0; s < kMaxStages; s++) {
            mbar_init(smem_u32(s_full + s), 1);
            mbar_init(smem_u32(s_empty + s), NCW);
            s_next[s] = 0;
        }
        mbar_fence_init();
    }
    if (tid < 64) {
        int nib = tid >> 2, r = tid & 3, pos = 0;
        for (int b = 0, seen = 0; b < 4; b++)
            if (nib & (1 << b)) { if (seen == r) pos = b; seen++; }
        s_sel[tid] = (uint8_t) pos;
    }
    // never-matching words below each stage: a candidate in the first row of a band whose shifted column is -1..-4
    if (tid < NSTG * kPrePad) s_stage[(tid / kPrePad) * stage_stride - kPrePad + (tid % kPrePad)] = CDS_CODE_PAD_WORD;
    __syncthreads();

    if (warp == NCW) {
        // ------------------------------------------------------------------ producer (one lane)
        // Drives the barriers and the bulk copies, and publishes with every stage the range of the group's word list that falls
        // into the band's rows (two reads of the group's row-start table), so consumers never meet at a CTA-wide barrier.
        if (lane == 0) {
            uint32_t q = 0;                 // running band number across items: stage = q % NSTG, use = q / NSTG
            int stage = 0;
            uint32_t use = 0;
            uint32_t iseq = 0;
            for (;;) {
                const long long w = (long long) atomicAdd(p.work_counter, 1ull);
                const bool done = w >= n_items;
                const int nb = done ? 1 : NB;
                const int64_t t = done ? 0 : w % p.n_targets;
                const uint32_t *gstart = done ? nullptr : p.groups[w / p.n_targets].gstart;
                for (int b = 0; b < nb; b++, q++, stage++) {
                    if (stage == NSTG) { stage = 0; use++; }
                    const int y0 = b * R;
                    const int y1 = min(y0 + R, H);
                    uint2 range = make_uint2(0u, 0u);
                    if (!done) range = make_uint2(__ldg(gstart + y0 / 4), __ldg(gstart + (y1 + 3) / 4));     // tile rows of the band; issued before the wait below
                    if (use > 0) mbar_wait(smem_u32(s_empty + stage), (use - 1) & 1);
                    if (trace && iseq < (uint32_t) kTraceItems) trace[(((size_t) iseq * kMaxBands + b) * 32 + 31) * 2] = clock64();
                    s_next[stage] = 0;
                    {
                        BandInfo bi;
                        bi.first = range.x; bi.end = range.y;
                        bi.band_lo = (uint32_t) ((y0 / 4) * rowpitch);
                        bi.band_hi = (uint32_t) (((y1 + 3) / 4) * rowpitch) - 1u;
                        bi.j_first = range.x >> 5;
                        bi.n_tk = range.y > range.x ? ((range.y - 1u) >> 5) - bi.j_first + 1u : 0u;
                        // a multiple of the number of consumer warps, so that every warp gets the same number of (partly filled) batches
                        bi.n_batches = (uint32_t) NCW * ((bi.n_tk + 32u * NCW - 1u) / (32u * NCW));
                        bi.pad = 0u;
                        s_band[stage] = bi;
                    }
                    if (b == 0) { s_item[2 * (iseq & 1)] = done ? -1 : t; s_item[2 * (iseq & 1) + 1] = done ? 0 : w / p.n_targets; }
                    const uint32_t bar = smem_u32(s_full + stage);
                    if (done) { mbar_arrive(bar); break; }
                    const uint32_t bytes = (uint32_t) ((y1 - y0 + 2 * S) * pitch) * 4u;
                    const uint32_t *src = p.planes + p.g.row_offset(t, 0) + (long long) (y0 - S) * pitch;   // guard rows cover y0 - S < 0
                    // the occupancy tile rows without their OR rows (which this kernel never reads), and without their band bytes when
                    // the filter is off (bitmaps built per chunk have none): one copy per tile row
                    const int n_trows = (y1 - y0 + 3) / 4;
                    const uint32_t rbytes = (uint32_t) (p.band_filter ? rowpitch : occupancy_band_offset(p.bpitch)) * 4u;
                    const uint32_t *bsrc = p.occ + ((size_t) t * occupancy_tile_rows(H) + y0 / 4) * occupancy_row_pitch(p.bpitch);
                    mbar_expect_tx(bar, bytes + (uint32_t) n_trows * rbytes);
                    if (HINT) bulk_load_hint(smem_u32(s_stage + (size_t) stage * stage_stride), src, bytes, bar, pol_stream);
                    else bulk_load(smem_u32(s_stage + (size_t) stage * stage_stride), src, bytes, bar);
                    for (int r = 0; r < n_trows; r++) {
                        const uint32_t dst = smem_u32(s_bits + (size_t) stage * bits_words + (size_t) r * rowpitch);
                        const uint32_t *rsrc = bsrc + (size_t) r * occupancy_row_pitch(p.bpitch);
                        if (HINT) bulk_load_hint(dst, rsrc, rbytes, bar, pol_stream);
                        else bulk_load(dst, rsrc, rbytes, bar);
                    }
                }
                if (done) break;
                iseq++;
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumers
    uint32_t iseq = 0;
    int stage = 0;                                   // stage and use count of the band this warp is at
    uint32_t use = 0;
    int cur_gi = -1;
    const uint4 *gwords = nullptr;                   // word list of the current group
    const uint16_t *glpal = nullptr;                 // palette references of its entries' set bits
    const uint32_t *gtocc = nullptr;                 // occupancy word of the first entry of every ticket of 32 entries
    uint2 *myq = s_queue + warp * kQueue;
    uint4 *mywq = s_wqueue + warp * kWordQueue;
    const uint32_t mywq_addr = smem_u32(mywq);
    const uint32_t lt_mask = (1u << lane) - 1u;
    const int *acc_base = s_acc;
    auto wait_full = [&]() {
        if (p.wait_mode == 0) mbar_wait(smem_u32(s_full + stage), use & 1);
        else mbar_wait_parked(smem_u32(s_full + stage), use & 1, p.wait_mode);
    };
    for (;;) {
        wait_full();
        const int64_t t = *reinterpret_cast<volatile long long *>(s_item + 2 * (iseq & 1));     // the producer did the 64-bit divisions
        if (t < 0) break;
        const int gi = (int) *reinterpret_cast<volatile long long *>(s_item + 2 * (iseq & 1) + 1);
        const int m0 = gi * GROUP;
        const int mb = min(GROUP, p.n_masks - m0);

        if (gi != cur_gi) {
            // per-group tables.  Every consumer passed the barrier that ends the previous item, so nobody still reads the old ones.
            const PaletteGroup pg = p.groups[m0 / CDS_PALETTE_GROUP];
            gwords = pg.words;
            glpal = pg.lpal;
            gtocc = pg.tocc;
            if (!WIDE) {
                for (int i = tid; i < pg.n_pal; i += NCT) s_pal[i] = pg.palette[i];
                if (tid == 0) s_pal[p.pal_entries - 1] = make_uint2(CDS_PAL_EMPTY_LO, CDS_PAL_EMPTY_LO);   // idle lanes point here
            }
            consumer_barrier<NCT>();
            cur_gi = gi;
        }

        for (int b = 0; b < NB; b++) {
            if (b > 0) wait_full();
            if (trace && iseq < (uint32_t) kTraceItems && lane == 0) trace[(((size_t) iseq * kMaxBands + b) * 32 + warp) * 2] = clock64();
            const uint32_t *band = s_stage + (size_t) stage * stage_stride;
            const int y0 = b * R;
            const volatile BandInfo *bi = s_band + stage;                      // read where needed: cheaper than six more live registers
            const uint2 range = make_uint2(bi->first, bi->end);                 // the group's word-list entries of this band

            uint32_t qh = 0, qt = 0;            // candidate queue head / tail (free running, slot = index & (kQueue - 1))
            uint32_t wcnt = 0;                  // words in the word queue
            // Both queues live for the whole band: words and candidates of different masks mix freely (they carry the mask's
            // index), so only the LAST batch of a band runs on a partly filled warp.

            // Peels the set bits of 32 queued words (one word per lane; `c` = 0 for idle lanes) into the candidate queue,
            // lowest bit first, one bit per lane per round, and evaluates whenever 32 candidates are waiting.
            // A full batch of candidates: start its palette-index loads, evaluate the batch submitted before it.
            const uint2 idle_cand = make_uint2((uint32_t) (S * pitch), 0u);      // an idle lane reads the band's first pixel and matches nothing
            uint2 pend_cand = idle_cand;
            uint32_t pend_pr = 0;
            bool pend = false;
            auto run_pending = [&]() { eval_candidates<NRINGS, WIDE>(pend_cand, pend_pr, band, pitch, s_pal, acc_base); };
            auto submit = [&](uint2 cand, bool live) {
                const uint32_t pr = fetch_palette_ref<WIDE>(cand, live, glpal, pol_keep, (uint32_t) p.pal_entries - 1u);
                if (pend) run_pending();
                pend_cand = cand; pend_pr = pr; pend = true;
            };
            // Turns the candidate bits `c` of 32 queued words (one word per lane, `e` its list entry; c = 0 for idle lanes) into
            // candidates, 32 per round, and evaluates them.
            auto peel = [&](uint32_t c, uint4 e) {          // e = {bits, -, lrec, meta} of the word's list entry
                const uint32_t wbits = e.x, lrec = e.z;
                // offset of the tile's first pixel inside the staged band | index of the (mask, orientation)'s first accumulator << 15;
                // a set bit adds (bit & 7) + (bit >> 3) * pitch
                const uint32_t base = (uint32_t) (((int) (e.w & 255u) * 4 - y0 + S) * pitch) + (((e.w >> kWordMetaColShift) & 255u) << 3) +
                                      (((e.w >> kWordMetaMaskShift) * (uint32_t) NVP + ((e.w >> kWordMetaOrientBit) & 1u) * (uint32_t) NS) << kCandOffsetBits);
                // Load-balanced expansion: the batch's T candidate bits are numbered word by word (prefix sums of the popcounts),
                // and in every round lane j takes candidate number j0 + j -- whichever word it belongs to -- so a round costs the
                // same whether the bits sit in one dense tile or are spread over all 32.
                const uint32_t n = (uint32_t) __popc(c);
                uint32_t incl = n;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += v;
                }
                const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
                const uint32_t excl = incl - n;
                for (uint32_t j0 = 0; j0 < total; j0 += 32) {
                    const uint32_t j = j0 + (uint32_t) lane;
                    // source word of candidate j = (number of words that start at or before j) - 1.  Every queued word has at
                    // least one candidate, so the words that START inside this round mark distinct bits of one 32-bit word
                    // (one OR-reduction), and a lane counts the marks at or below its own position.
                    const uint32_t rel = excl - j0;
                    const uint32_t starts = __reduce_or_sync(0xffffffffu, rel < 32u ? 1u << rel : 0u);
                    const uint32_t w_first = (uint32_t) __popc(__ballot_sync(0xffffffffu, excl < j0));     // words that started in earlier rounds
                    uint32_t src = w_first + (uint32_t) __popc(starts & (lt_mask + lt_mask + 1u)) - 1u;
                    const bool live = j < total;
                    src &= 31u;
                    const uint32_t cs = __shfl_sync(0xffffffffu, c, (int) src), es = __shfl_sync(0xffffffffu, excl, (int) src);
                    const uint32_t bs = __shfl_sync(0xffffffffu, base, (int) src), ls = __shfl_sync(0xffffffffu, lrec, (int) src);
                    const uint32_t ws = __shfl_sync(0xffffffffu, wbits, (int) src);
                    uint2 cand = idle_cand;
                    if (live) {
                        const uint32_t bit = select_bit(cs, j - es, s_sel);              // the (j - es)-th candidate bit of that word
                        cand.x = bs + (bit & 7u) + (bit >> 3) * (uint32_t) pitch;
                        cand.y = ls + (uint32_t) __popc(ws & ((1u << bit) - 1u));
                    }
                    if (j0 + 32 <= total) {
                        submit(cand, true);                                             // a full round goes straight to evaluation
                    } else {
                        // the batch's last, partial round waits in the candidate queue for company
                        if (live) myq[(qt + (uint32_t) lane) & (kQueue - 1)] = cand;
                        qt += total - j0;
                        if (qt - qh >= 32) {
                            __syncwarp();
                            const uint2 full = myq[(qh + lane) & (kQueue - 1)];
                            qh += 32;
                            submit(full, true);
                        }
                    }
                }
            };
            // The queued words (at most 32, one per lane) are expanded and evaluated.  The queue holds everything the expansion needs
            // of a word's entry, so nothing is read again (round 1 queued {bits, entry index} and re-read the entries a batch later).
            auto drain_words = [&]() {
                __syncwarp();
                uint4 e = make_uint4(0u, 0u, 0u, 0u);
                if (lane < (int) wcnt) e = mywq[lane];
                wcnt = 0;
                __syncwarp();                                           // the slots may be written again
                peel(e.x, make_uint4(e.y, 0u, e.z, e.w));
            };

            // Tickets.  Inside a tile row the entries are ordered by occupancy word (sector, tile column), so the 32 entries of
            // a ticket (entries 32 j .. 32 j + 31 of the list) concern the contiguous run of occupancy words between the first
            // entry of this ticket and the first entry of the next one (pg.tocc, one word per ticket).  On colour-depth MIPs
            // ~97 % of the entries sit on tiles where the target has nothing in that sector, so a warp first TESTS 32 tickets,
            // one per lane -- is any occupancy word of the ticket's run set? -- and then scans only the tickets that passed.
            // Tickets are dealt out strided (lane i of batch b gets ticket b + i * n_batches): neighbouring tickets, which tend
            // to pass or fail together, go to different warps.
            const uint32_t band_lo = bi->band_lo;
            const uint32_t *bits_y0 = s_bits + (size_t) stage * bits_words - band_lo;          // indexed by the entries' absolute occupancy word index
            const uint32_t sec_words = (uint32_t) (CDS_NUM_SECTORS * p.bpitch);
            const uint32_t nz_off = (uint32_t) occupancy_nz_offset(p.bpitch);        // the non-empty bits of a tile row, behind its sector rows
            const uint4 idle = make_uint4(0u, band_lo, 0u, 0u);
            auto scan_one = [&](uint4 w) {
                const uint32_t occ_i = w.y & kWordOccMask;
                uint32_t c = w.x & bits_y0[occ_i];                      // mask pixels of this word that can match
                // Rank-band filter.  The tile's byte holds the band of every target pixel that any shifted variant of any pixel of
                // the tile can read in this sector, the entry's byte every band that one of its pixels' intervals (in this sector)
                // touches.  A pixel matches a target pixel only when that pixel's rank lies in its interval, and then both bytes
                // share that rank's band; disjoint bytes therefore mean that no pixel of the word can match in any variant, and
                // dropping the word changes no count.  The byte of word i of tile row ty is byte i - ty * rowpitch of the row's
                // band words, i.e. byte i + ty * 3 rowpitch + 4 * band offset counted from bits_y0.
                if (c && p.band_filter) {
                    const uint32_t bi = occ_i + (w.w & 255u) * (3u * (uint32_t) rowpitch) + 4u * (uint32_t) occupancy_band_offset(p.bpitch);
                    const uint32_t tb = reinterpret_cast<const uint8_t *>(bits_y0)[bi];
                    if ((tb & (w.y >> kWordBandShift)) == 0u) c = 0u;
                }
                // words with candidates are compacted first, so that the bit expansion runs on (nearly) full warps: when the new ones
                // do not fit behind the queued ones, those are expanded first
                const unsigned has = __ballot_sync(0xffffffffu, c != 0);
                const uint32_t n_new = (uint32_t) __popc(has);
                if (wcnt + n_new > (uint32_t) kWordQueue) drain_words();
                if (c) {
                    const uint32_t slot = wcnt + (uint32_t) __popc(has & lt_mask);
                    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(mywq_addr + slot * 16u), "r"(c), "r"(w.x), "r"(w.z), "r"(w.w) : "memory");
                }
                wcnt += n_new;
            };
            auto load = [&](uint32_t jt) -> uint4 {                     // this lane's entry of ticket jt
                const uint32_t i = (jt << 5) + (uint32_t) lane;
                uint4 w = idle;
                if (i >= range.x && i < range.y) w = HINT ? ldg_hint_v4(gwords + i, pol_keep) : __ldg(gwords + i);
                return w;
            };
            for (;;) {
                uint32_t bt = 0;
                if (lane == 0) bt = (uint32_t) atomicAdd(&s_next[stage], 1);
                bt = __shfl_sync(0xffffffffu, bt, 0);
                const uint32_t n_batches = bi->n_batches;
                if (bt >= n_batches || p.debug_skip) break;
                const uint32_t k = bt + (uint32_t) lane * n_batches;
                const uint32_t jt = bi->j_first + k;
                bool pass = false;
                if (k < bi->n_tk) {
                    // tickets cut by the band's ends take the band's bound (their neighbours belong to other tile rows)
                    const uint32_t band_hi = bi->band_hi;
                    uint32_t o_lo = band_lo, o_hi = band_hi;
                    if ((jt << 5) >= range.x) o_lo = max(band_lo, HINT ? ldg_hint_u32(gtocc + jt, pol_keep) : __ldg(gtocc + jt));
                    if (((jt + 1u) << 5) < range.y) o_hi = min(band_hi, HINT ? ldg_hint_u32(gtocc + jt + 1u, pol_keep) : __ldg(gtocc + jt + 1u));
                    if (!p.ticket_skip) {
                        pass = true;
                    } else {
                        // the run [o_lo, o_hi], tile row by tile row, against the rows' non-empty bits (one bit per sector word,
                        // cds_kernels.cuh): a few masked words instead of a walk over the occupancy words themselves
                        uint32_t ra = o_lo - band_lo, base = band_lo;
                        while (ra >= (uint32_t) rowpitch) { ra -= (uint32_t) rowpitch; base += (uint32_t) rowpitch; }
                        uint32_t re = o_hi - base;                       // may lie in a later tile row
                        for (;;) {
                            const uint32_t hi = min(re, sec_words - 1u);
                            if (ra <= hi) {
                                const uint32_t *nz = bits_y0 + base + nz_off;
                                for (uint32_t wd = ra >> 5; wd <= (hi >> 5); wd++) {
                                    uint32_t m = nz[wd];
                                    if (wd == (ra >> 5)) m &= 0xffffffffu << (ra & 31u);
                                    if (wd == (hi >> 5)) m &= 0xffffffffu >> (31u - (hi & 31u));
                                    pass |= m != 0u;
                                }
                            }
                            if (re < (uint32_t) rowpitch) break;
                            re -= (uint32_t) rowpitch; base += (uint32_t) rowpitch; ra = 0;
                        }
                    }
                }
                unsigned live = __ballot_sync(0xffffffffu, pass);
                if (!live) continue;
                // scan the tickets that passed; the next one's entries are requested before the current one is used
                int src = __ffs((int) live) - 1;
                live &= live - 1;
                uint32_t jc = __shfl_sync(0xffffffffu, jt, src);
                // (two tickets per trip, in two sets of registers: a single set would need the requested entries MOVED into the scanned
                // ones, and a move waits for the load -- the request would hide nothing)
                uint4 wa = load(jc), wb = idle;
                for (;;) {
                    bool more = live != 0;
                    if (more) {
                        src = __ffs((int) live) - 1;
                        live &= live - 1;
                        jc = __shfl_sync(0xffffffffu, jt, src);
                        wb = load(jc);
                    }
                    scan_one(wa);
                    if (!more) break;
                    more = live != 0;
                    if (more) {
                        src = __ffs((int) live) - 1;
                        live &= live - 1;
                        jc = __shfl_sync(0xffffffffu, jt, src);
                        wa = load(jc);
                    }
                    scan_one(wb);
                    if (!more) break;
                }
            }
            // the band's last, partly filled batches: everything queued reads this stage, so it is evaluated before the release
            if (wcnt) drain_words();
            if (qt != qh) {
                __syncwarp();
                const bool live = lane < (int) (qt - qh);
                uint2 cand = idle_cand;
                if (live) cand = myq[(qh + lane) & (kQueue - 1)];
                submit(cand, live);
            }
            if (pend) run_pending();
            // this warp is done with the stage: let the producer refill it
            __syncwarp();
            if (trace && iseq < (uint32_t) kTraceItems && lane == 0) trace[(((size_t) iseq * kMaxBands + b) * 32 + warp) * 2 + 1] = clock64();
            if (lane == 0) mbar_arrive(smem_u32(s_empty + stage));
            if (++stage == NSTG) { stage = 0; use++; }
        }

        // item epilogue: max over variants per orientation; mirrored wins only when strictly greater
        __threadfence();                    // this thread's reductions are performed before anybody reads the accumulators
        consumer_barrier<NCT>();
        for (int mi = tid; mi < mb; mi += NCT) {
            // a mask's counters as whole 16-byte words; most masks have no hit at all on most targets, and then nothing is written back
            int4 *a4 = reinterpret_cast<int4 *>(s_acc + mi * NVP);
            int a[NVP];
#pragma unroll
            for (int v = 0; v < NVP / 4; v++) {
                const int4 q4 = __ldcg(a4 + v);
                a[4 * v] = q4.x; a[4 * v + 1] = q4.y; a[4 * v + 2] = q4.z; a[4 * v + 3] = q4.w;
            }
            int best = 0, bestm = 0;
#pragma unroll
            for (int v = 0; v < NS; v++) best = max(best, a[v]);
#pragma unroll
            for (int v = 0; v < NS; v++) bestm = max(bestm, a[NS + v]);
            int word = best;
            if (bestm > best) word = bestm | CDS_SCORE_MIRROR_BIT;          // no mirrored words in the lists -> bestm stays 0
            p.scores[(size_t) (m0 + mi) * p.n_targets + t] = word;
            if ((best | bestm) != 0) {
#pragma unroll
                for (int v = 0; v < NVP / 4; v++) __stcg(a4 + v, make_int4(0, 0, 0, 0));
            }
        }
        consumer_barrier<NCT>();
        iseq++;
    }
}

struct CandConfig {
    int rows_per_band, n_bands, stage_words;
    size_t smem_bytes;
    bool ok;
};

// `pal_entries`: palette entries staged (cand_staged_palette)
template <int GROUP>
CandConfig cand_config(int xy_shift, const PlaneGeom &g, int n_warps, int n_stages, int max_rows, int pal_entries)
{
    const int bpitch = occupancy_tile_pitch(g.W);
    CandConfig c{};
    const int S = xy_shift;
    const int NS = xy_shift == 0 ? 1 : (xy_shift == 2 ? 9 : 17);
    const size_t budget = 227 * 1024;
    int R_top = (g.H + 3) / 4 * 4;
    if (max_rows >= 4) R_top = std::min(R_top, max_rows / 4 * 4);
    for (int R = R_top; R >= 4; R -= 4) {        // whole occupancy tiles per band
        int n_bands = (g.H + R - 1) / R;
        if (n_bands > kMaxBands) break;
        size_t stage_words = (size_t) (R + 2 * S) * g.pitch;
        if (stage_words >= (1u << kCandOffsetBits)) continue;       // candidates address the band with kCandOffsetBits bits (and a bulk copy stays below 1 MB)
        CandSmem<GROUP> L((int) stage_words, NS, (R / 4) * occupancy_stage_pitch(bpitch), n_warps, n_stages, pal_entries);
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
               const uint32_t *occ, int bpitch, const PaletteGroup *groups, int xy_shift, int32_t *scores,
               const MatchScratch &scratch, cudaStream_t s, int dev, bool wide, bool band_bytes, int pal_entries)
{
    const int n_stages = std::max(2, std::min(kMaxStages, cand_tuning().stages));
    CandConfig c = cand_config<GROUP>(xy_shift, g, NCW, n_stages, cand_tuning().max_rows, pal_entries);
    if (!c.ok) return 0;
    CandParams p;
    p.masks = masks; p.n_masks = n_masks; p.planes = planes; p.g = g; p.n_targets = n_targets; p.scores = scores;
    p.work_counter = scratch.work_counter;
    p.acc = scratch.acc;
    p.rows_per_band = c.rows_per_band; p.n_bands = c.n_bands; p.stage_words = c.stage_words;
    p.n_groups = (n_masks + GROUP - 1) / GROUP;
    p.occ = occ; p.bpitch = bpitch; p.groups = groups;
    static const int debug_skip = env_int("CDSGPU_CAND_NULL", 0);
    p.debug_skip = debug_skip;
    static const int no_skip = env_int("CDSGPU_CAND_NOSKIP", 0);
    p.ticket_skip = no_skip ? 0 : 1;
    p.wait_mode = cand_tuning().wait_mode;
    p.n_stages = n_stages;
    p.band_filter = band_bytes && !env_int("CDSGPU_CAND_NOBAND", 0);   // read at every launch: tests compare both settings in one process
    p.pal_entries = pal_entries;
    const int hint = cand_tuning().l2_hint;
    static const char *trace_path = std::getenv("CDSGPU_CAND_TRACE");
    p.trace = nullptr;
    const size_t trace_bytes = (size_t) kTraceItems * kMaxBands * 32 * 2 * sizeof(long long);
    if (trace_path) {
        cudaMalloc(&p.trace, trace_bytes);
        cudaMemsetAsync(p.trace, 0, trace_bytes, s);
    }
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    long long n_items = (long long) p.n_groups * n_targets;
    int grid = (int) std::min<long long>(std::min(n_sm, 256), n_items);
    void (*kern)(const CandParams) = nullptr;
    const int rings = xy_shift / 2;
    if (wide) {
        if (rings == 0) kern = pixelmatch_cand_kernel<0, GROUP, NCW, false, true>;
        else if (rings == 1) kern = pixelmatch_cand_kernel<1, GROUP, NCW, false, true>;
        else kern = pixelmatch_cand_kernel<2, GROUP, NCW, false, true>;
    } else if (rings == 0) kern = pixelmatch_cand_kernel<0, GROUP, NCW, false, false>;
    else if (rings == 1) kern = hint ? pixelmatch_cand_kernel<1, GROUP, NCW, true, false> : pixelmatch_cand_kernel<1, GROUP, NCW, false, false>;
    else kern = pixelmatch_cand_kernel<2, GROUP, NCW, false, false>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) c.smem_bytes);
    kern<<<grid, (NCW + 1) * 32, c.smem_bytes, s>>>(p);
    if (p.trace) {
        // profiling aid: dump the clocks (this synchronises the stream)
        std::vector<long long> h(trace_bytes / sizeof(long long));
        cudaStreamSynchronize(s);
        cudaMemcpy(h.data(), p.trace, trace_bytes, cudaMemcpyDeviceToHost);
        cudaFree(p.trace);
        if (FILE *f = std::fopen(trace_path, "wb")) {
            const int hdr[4] = {kTraceItems, kMaxBands, c.n_bands, NCW};
            std::fwrite(hdr, sizeof hdr, 1, f);
            std::fwrite(h.data(), 1, trace_bytes, f);
            std::fclose(f);
        }
    }
    return 1;
}

// ------------------------------------------------------------------------------------------------------------------
// Word lists.  One warp per (mask, row): the row's records are scattered into two shared-memory bitmaps (unmirrored and
// mirrored target coordinates), whose non-zero words become the entries.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kRowTiles = 256;      // W <= 2048: tile columns per tile row
constexpr int kLists = 2 * CDS_NUM_SECTORS;      // (orientation, sector) bitmaps per mask tile row

// Rank bands (occupancy_rank_band) that an interval [lo, lo + len] (SR units) touches, as a byte; 0 for an empty interval.
__device__ __forceinline__ uint32_t interval_band_byte(uint32_t lo, uint32_t len)
{
    if (lo == CDS_IV_EMPTY) return 0u;
    const uint32_t r0 = lo % CDS_SECTOR_STRIDE, r1 = min(r0 + len, (uint32_t) CDS_NUM_RANKS - 1u);
    return (2u << occupancy_rank_band(r1)) - (1u << occupancy_rank_band(r0));
}

// Scatters the records of one mask TILE ROW (4 image rows) into the (orientation, sector) tile bitmaps: pixel (x, y) is bit
// (y % 4) * 8 + (x % 8) of tile word x / 8.  A mask pixel goes into the list of the sector of each of its non-empty rank
// intervals: its own sector (interval 1) and, near a sector boundary, one neighbouring sector (interval 2).  `pix` (may be null)
// receives, per (y % 4, x), the pixel's palette index | own sector << 11 | band byte of interval 1 << 16 | of interval 2 << 24.
__device__ __forceinline__ void build_tile_row_lists(const MaskDesc &md, int ty, int W, int H, bool mirror,
                                                     const cds_class_interval *__restrict__ class_tab,
                                                     uint32_t (*bm)[kRowTiles] /* [kLists] */, uint32_t *pix, uint32_t *pix_cls = nullptr)
{
    const int lane = threadIdx.x & 31;
    for (int k = lane; k < kLists * kRowTiles; k += 32) bm[0][k] = 0;
    __syncwarp();
    const uint32_t r0 = __ldg(md.rowstart + 4 * ty), r1 = __ldg(md.rowstart + min(4 * ty + 4, H));
    for (uint32_t i = r0 + lane; i < r1; i += 32) {
        const uint32_t cls = __ldg(md.classes + i);
        if (cls >= (uint32_t) CDS_NUM_CLASSES) continue;                       // no colour sector: matches nothing
        const uint32_t xy = __ldg(&md.records[i].xy);
        const int x = (int) (xy & 0xFFFFu), yy = (int) (xy >> 16) & 3;
        const int xm = W - 1 - x;
        const int s1 = (int) (cls / CDS_NUM_RANKS);
        const cds_class_interval iv = class_tab[cls];
        if (pix) pix[yy * (kRowTiles * 8) + x] = (md.crec ? (__ldg(md.crec + i) >> 21) : 0u) | ((uint32_t) s1 << 11) |
                                                  (interval_band_byte(iv.lo1, iv.len1) << 16) | (interval_band_byte(iv.lo2, iv.len2) << 24);
        if (pix_cls) pix_cls[yy * (kRowTiles * 8) + x] = cls;
        const uint32_t bn = 1u << (yy * 8 + (x & 7)), bmr = 1u << (yy * 8 + (xm & 7));
        if (iv.lo1 != CDS_IV_EMPTY) {
            atomicOr(&bm[s1][x >> 3], bn);
            if (mirror) atomicOr(&bm[CDS_NUM_SECTORS + s1][xm >> 3], bmr);
        }
        if (iv.lo2 != CDS_IV_EMPTY) {
            const int s2 = (int) (iv.lo2 / CDS_SECTOR_STRIDE);
            atomicOr(&bm[s2][x >> 3], bn);
            if (mirror) atomicOr(&bm[CDS_NUM_SECTORS + s2][xm >> 3], bmr);
        }
    }
    __syncwarp();
}

// counts[m][ty] = {word-list entries, set bits} of (mask m, tile row ty); one warp per (mask, tile row)
__global__ void __launch_bounds__(32) words_count_kernel(const MaskDesc *__restrict__ masks, int W, int H, bool mirror,
                                                         const cds_class_interval *__restrict__ class_tab,
                                                         uint32_t *__restrict__ wcount, uint32_t *__restrict__ bcount)
{
    __shared__ uint32_t s_bm[kLists][kRowTiles];
    const int lane = threadIdx.x;
    const int ty = blockIdx.x, HT = gridDim.x;
    const int m = blockIdx.y;
    const MaskDesc md = masks[m];
    build_tile_row_lists(md, ty, W, H, mirror, class_tab, s_bm, nullptr);
    int nw = 0, nb = 0;
    for (int k = lane; k < kLists * kRowTiles; k += 32) {
        const uint32_t wbits = s_bm[0][k];
        nw += wbits != 0;
        nb += __popc(wbits);
    }
    nw = __reduce_add_sync(0xffffffffu, nw);
    nb = __reduce_add_sync(0xffffffffu, nb);
    if (lane == 0) {
        wcount[(size_t) m * (HT + 1) + ty] = (uint32_t) nw;
        bcount[(size_t) m * (HT + 1) + ty] = (uint32_t) nb;
    }
}

// For every (group, row): the totals of the group's masks in that row (grow), and for every mask its offset inside that run
// (in place over the per-mask counts).  Run twice: for the entry counts and for the bit counts.
__global__ void __launch_bounds__(128) words_group_rows_kernel(uint32_t *__restrict__ count /* [M][H+1] counts -> offsets */, int n_masks, int H,
                                                                uint32_t *__restrict__ grow /* [n_groups][H+1] */)
{
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    const int g = blockIdx.y;
    if (y >= H) return;
    uint32_t acc = 0;
    const int m1 = min(n_masks, (g + 1) * CDS_PALETTE_GROUP);
    for (int m = g * CDS_PALETTE_GROUP; m < m1; m++) {
        const size_t i = (size_t) m * (H + 1) + y;
        const uint32_t c = count[i];
        count[i] = acc;
        acc += c;
    }
    grow[(size_t) g * (H + 1) + y] = acc;
}

// one interval as a palette word (cds_common.h): lo | len << 18, SR units
__device__ __forceinline__ uint32_t pack_interval_word(uint32_t lo, uint32_t len)
{
    if (lo == CDS_IV_EMPTY || len > CDS_PAL_MAX_LEN) return CDS_PAL_EMPTY_LO;
    return lo | (len << CDS_PAL_LO_BITS);
}

template <bool WIDE>
__global__ void __launch_bounds__(32) words_fill_kernel(const MaskDesc *__restrict__ masks, int first_mask, int W, int H, bool mirror,
                                                        const cds_class_interval *__restrict__ class_tab,
                                                        const uint32_t *__restrict__ gstart /* [n_groups][HT+1] entries */,
                                                        const uint32_t *__restrict__ bstart /* [n_groups][HT+1] bits */,
                                                        const uint32_t *__restrict__ boff /* [M][HT+1] */,
                                                        uint4 *__restrict__ words, uint16_t *__restrict__ lpal)
{
    __shared__ uint32_t s_bm[kLists][kRowTiles];
    // per (y % 4, x): palette index | own sector << 11 | the intervals' band bytes << 16, << 24, or (WIDE) the pixel's colour class
    __shared__ uint32_t s_pix[4 * kRowTiles * 8];
    const int lane = threadIdx.x;
    const int ty = blockIdx.x, HT = gridDim.x;
    const int m = first_mask + blockIdx.y;
    const MaskDesc md = masks[blockIdx.y];
    if constexpr (WIDE) build_tile_row_lists(md, ty, W, H, mirror, class_tab, s_bm, nullptr, s_pix);
    else build_tile_row_lists(md, ty, W, H, mirror, class_tab, s_bm, s_pix);
    const int g = m / CDS_PALETTE_GROUP;
    const uint32_t mtag = (uint32_t) (m % CDS_PALETTE_GROUP) << kWordMetaMaskShift;
    uint32_t out_w = __ldg(gstart + (size_t) g * (HT + 1) + ty) + __ldg(md.wstart + ty);       // start of the tile row's run + this mask's offset in it
    uint32_t out_b = __ldg(bstart + (size_t) g * (HT + 1) + ty) + __ldg(boff + (size_t) m * (HT + 1) + ty);
    const uint32_t lt = (1u << lane) - 1u;
    const int tp = occupancy_tile_pitch(W);
    const int n_tiles = (W + 7) / 8;
    for (int list = 0; list < (mirror ? kLists : CDS_NUM_SECTORS); list++) {
        const int o = list / CDS_NUM_SECTORS, sec = list % CDS_NUM_SECTORS;
        for (int k0 = 0; k0 < n_tiles; k0 += 32) {
            const int k = k0 + lane;
            uint32_t wbits = k < kRowTiles ? s_bm[list][k] : 0u;
            const unsigned bal = __ballot_sync(0xffffffffu, wbits != 0);
            if (bal == 0) continue;
            const uint32_t pc = (uint32_t) __popc(wbits);
            uint32_t incl = pc;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += v;
            }
            if (wbits) {
                const uint32_t pos = out_w + (uint32_t) __popc(bal & lt);
                uint32_t lrec = out_b + incl - pc;
                const uint4 e = make_uint4(wbits, (uint32_t) (ty * occupancy_stage_pitch(tp) + sec * tp + k), lrec,
                                           (uint32_t) ty | ((uint32_t) k << kWordMetaColShift) | ((uint32_t) o << kWordMetaOrientBit) |
                                               ((uint32_t) sec << kWordMetaSectorShift) | mtag);
                uint32_t bands = 0u;        // the word's rank-band byte: OR over its pixels of the bands of their interval in this sector
                // palette references of the word's pixels, in bit order: index | (interval 2 ? 0x8000 : 0)
                while (wbits) {
                    const int bit = __ffs((int) wbits) - 1;
                    wbits &= wbits - 1;
                    const int xt = k * 8 + (bit & 7);
                    const uint32_t pv = s_pix[(bit >> 3) * (kRowTiles * 8) + (o ? W - 1 - xt : xt)];
                    if constexpr (WIDE) {
                        // the interval of this list's sector, packed like a palette word (cds_common.h)
                        const cds_class_interval iv = class_tab[pv];
                        const bool own = pv / CDS_NUM_RANKS == (uint32_t) sec;
                        reinterpret_cast<uint32_t *>(lpal)[lrec++] = pack_interval_word(own ? iv.lo1 : iv.lo2, own ? iv.len1 : iv.len2);
                        bands |= interval_band_byte(own ? iv.lo1 : iv.lo2, own ? iv.len1 : iv.len2);
                    } else {
                        const bool own = ((pv >> 11) & 7u) == (uint32_t) sec;
                        lpal[lrec++] = (uint16_t) ((pv & 0x7FFu) | (own ? 0u : 0x8000u));
                        bands |= (pv >> (own ? 16 : 24)) & 0xFFu;
                    }
                }
                words[pos] = make_uint4(e.x, e.y | (bands << kWordBandShift), e.z, e.w);
            }
            out_w += (uint32_t) __popc(bal);
            out_b += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Bucket order.  words_fill_kernel writes a tile row's entries mask by mask; the kernel wants them ordered by occupancy word
// (sector, tile column) so that the entries that meet one target tile are neighbours and whole tickets can be skipped.
// A counting sort per group over the occupancy word index: count, exclusive scan, scatter (the order inside a bucket is
// whatever the atomics give -- scores are sums, they do not depend on it).
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) words_bucket_count_kernel(const uint4 *__restrict__ words, const uint32_t *__restrict__ gstart, int HT,
                                                                 uint32_t n_buckets, uint32_t *__restrict__ counts)
{
    const int g = blockIdx.y;
    const uint32_t e0 = gstart[(size_t) g * (HT + 1)], e1 = gstart[(size_t) g * (HT + 1) + HT];
    for (uint32_t i = e0 + blockIdx.x * blockDim.x + threadIdx.x; i < e1; i += gridDim.x * blockDim.x)
        atomicAdd(&counts[(size_t) g * n_buckets + (words[i].y & kWordOccMask)], 1u);
}

// one CTA per group: counts -> first entry of every bucket (absolute index), in place
__global__ void __launch_bounds__(1024) words_bucket_scan_kernel(uint32_t *__restrict__ counts, const uint32_t *__restrict__ gstart, int HT, uint32_t n_buckets)
{
    __shared__ uint32_t s_sum[1024];
    const int g = blockIdx.x;
    uint32_t *c = counts + (size_t) g * n_buckets;
    const uint32_t per = (n_buckets + 1023u) / 1024u;
    const uint32_t b0 = min(threadIdx.x * per, n_buckets), b1 = min(b0 + per, n_buckets);
    uint32_t sum = 0;
    for (uint32_t b = b0; b < b1; b++) sum += c[b];
    s_sum[threadIdx.x] = sum;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const uint32_t v = threadIdx.x >= (unsigned) d ? s_sum[threadIdx.x - d] : 0u;
        __syncthreads();
        s_sum[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t acc = gstart[(size_t) g * (HT + 1)] + s_sum[threadIdx.x] - sum;
    for (uint32_t b = b0; b < b1; b++) { const uint32_t n = c[b]; c[b] = acc; acc += n; }
}

__global__ void __launch_bounds__(256) words_bucket_scatter_kernel(const uint4 *__restrict__ words, const uint32_t *__restrict__ gstart, int HT,
                                                                   uint32_t n_buckets, const uint32_t *__restrict__ first, uint32_t *__restrict__ cursor,
                                                                   uint4 *__restrict__ sorted)
{
    const int g = blockIdx.y;
    const uint32_t e0 = gstart[(size_t) g * (HT + 1)], e1 = gstart[(size_t) g * (HT + 1) + HT];
    for (uint32_t i = e0 + blockIdx.x * blockDim.x + threadIdx.x; i < e1; i += gridDim.x * blockDim.x) {
        const uint4 e = words[i];
        const size_t b = (size_t) g * n_buckets + (e.y & kWordOccMask);
        sorted[first[b] + atomicAdd(&cursor[b], 1u)] = e;
    }
}

// tocc[j] = occupancy word of entry 32 j (of the last entry beyond the end): the bounds of the tickets' occupancy runs
__global__ void __launch_bounds__(256) words_tocc_kernel(const uint4 *__restrict__ words, uint32_t n_entries, uint32_t n_tocc, uint32_t *__restrict__ tocc)
{
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_tocc) return;
    tocc[j] = n_entries ? words[min(j << 5, n_entries - 1u)].y & kWordOccMask : 0u;
}

}  // namespace

CandTuning &cand_tuning()
{
    // Waits poll try_wait by default.  Measured (profiles/r02_cand_trace.txt, tools/cand_sweep.py): a suspend-time hint does not stop the
    // hardware from returning at once, and sleeping between polls (32..400 ns) costs 1-3 % of the throughput without lowering the
    // instruction count -- the polling loop runs in issue slots that are idle anyway.
    static CandTuning t{env_int("CDSGPU_CAND_WAIT", 0), env_int("CDSGPU_CAND_L2HINT", 0), env_int("CDSGPU_CAND_WARPS", 31),
                        env_int("CDSGPU_CAND_STAGES", 2), env_int("CDSGPU_CAND_ROWS", 0)};
    return t;
}

void launch_words_tocc(const uint4 *words, uint32_t n_entries, uint32_t *tocc, cudaStream_t s)
{
    const uint32_t n = words_tocc_count(n_entries);
    words_tocc_kernel<<<(n + 255) / 256, 256, 0, s>>>(words, n_entries, n, tocc);
}

void launch_words_bucket_sort(const uint4 *words, const uint32_t *gstart, int n_groups, int W, int H, uint32_t *tables /* 2 * n_groups * buckets */,
                              uint4 *sorted, cudaStream_t s)
{
    if (n_groups == 0) return;
    const int HT = occupancy_tile_rows(H);
    const uint32_t nb = (uint32_t) words_bucket_count(W, H);
    uint32_t *first = tables, *cursor = tables + (size_t) n_groups * nb;
    cudaMemsetAsync(tables, 0, (size_t) 2 * n_groups * nb * sizeof(uint32_t), s);
    dim3 grid(148 * 4, n_groups);
    words_bucket_count_kernel<<<grid, 256, 0, s>>>(words, gstart, HT, nb, first);
    words_bucket_scan_kernel<<<n_groups, 1024, 0, s>>>(first, gstart, HT, nb);
    words_bucket_scatter_kernel<<<grid, 256, 0, s>>>(words, gstart, HT, nb, first, cursor, sorted);
}

bool cand_kernel_supported(int xy_shift, const PlaneGeom &g)
{
    static const bool disabled = std::getenv("CDSGPU_DISABLE_CAND") != nullptr;
    if (disabled) return false;
    if (!(xy_shift == 0 || xy_shift == 2 || xy_shift == 4)) return false;
    if (xy_shift > g.guard || xy_shift > g.pitch - g.W || xy_shift > kPrePad) return false;
    if (g.W > 2048 || g.H > 1024) return false;
    // word-list entries carry the occupancy word index in 24 bits (their rank-band byte above it)
    if ((size_t) occupancy_tile_rows(g.H) * occupancy_stage_pitch(occupancy_tile_pitch(g.W)) > kWordOccMask) return false;
    return cand_config<CDS_PALETTE_GROUP>(xy_shift, g, 16, 2, 0, CDS_PALETTE_SIZE).ok;      // whatever the palettes of a later launch
}

void launch_words_count(const MaskDesc *masks, int n_masks, int W, int H, bool mirror, const cds_class_interval *class_tab,
                        uint32_t *wcount, uint32_t *bcount, cudaStream_t s)
{
    for (int m0 = 0; m0 < n_masks; m0 += 32768) {
        int cnt = n_masks - m0 < 32768 ? n_masks - m0 : 32768;
        const int HT = occupancy_tile_rows(H);
        dim3 grid(HT, cnt);
        words_count_kernel<<<grid, 32, 0, s>>>(masks + m0, W, H, mirror, class_tab, wcount + (size_t) m0 * (HT + 1), bcount + (size_t) m0 * (HT + 1));
    }
}

void launch_words_group_rows(uint32_t *count, int n_masks, int H, uint32_t *grow, cudaStream_t s)
{
    const int n_groups = (n_masks + CDS_PALETTE_GROUP - 1) / CDS_PALETTE_GROUP;
    if (n_groups == 0) return;
    dim3 grid((H + 127) / 128, n_groups);
    words_group_rows_kernel<<<grid, 128, 0, s>>>(count, n_masks, H, grow);
}

void launch_words_fill(const MaskDesc *masks, int n_masks, int W, int H, bool mirror, const cds_class_interval *class_tab,
                       const uint32_t *gstart, const uint32_t *bstart, const uint32_t *boff, uint4 *words, uint16_t *lpal, cudaStream_t s,
                       bool wide_lpal)
{
    for (int m0 = 0; m0 < n_masks; m0 += 32768) {
        int cnt = n_masks - m0 < 32768 ? n_masks - m0 : 32768;
        dim3 grid(occupancy_tile_rows(H), cnt);
        if (wide_lpal) words_fill_kernel<true><<<grid, 32, 0, s>>>(masks + m0, m0, W, H, mirror, class_tab, gstart, bstart, boff, words, lpal);
        else words_fill_kernel<false><<<grid, 32, 0, s>>>(masks + m0, m0, W, H, mirror, class_tab, gstart, bstart, boff, words, lpal);
    }
}

CandShape cand_launch_shape(int xy_shift, const PlaneGeom &g, int pal_entries)
{
    // tuning knob (default picked from profiles/): consumer warps per CTA.  More warps need more
    // shared memory for their queues; when the band stages no longer fit (xyShift 4: 34 accumulators per mask) fewer are used.
    const int n_stages = std::max(2, std::min(kMaxStages, cand_tuning().stages));
    const int staged = cand_staged_palette(pal_entries);
    auto fits = [&](int w) { return cand_config<CDS_PALETTE_GROUP>(xy_shift, g, w, n_stages, cand_tuning().max_rows, staged); };
    int warps = cand_tuning().warps;
    if (warps >= 31 && !fits(31).ok) warps = 28;
    if (warps >= 28 && !fits(28).ok) warps = 24;
    if (warps >= 24 && !fits(24).ok) warps = 16;
    warps = warps >= 31 ? 31 : warps >= 28 ? 28 : warps >= 24 ? 24 : 16;
    const CandConfig c = fits(warps);
    return CandShape{warps, c.rows_per_band, n_stages, c.smem_bytes, c.ok};
}

int launch_pixelmatch_cand(const MaskDesc *masks, int n_masks, const uint32_t *planes, PlaneGeom g, int64_t n_targets,
                           const uint32_t *occ, int bpitch, const PaletteGroup *groups, int xy_shift, bool mirror,
                           int32_t *scores, const MatchScratch &scratch, cudaStream_t s, bool wide_lpal, bool band_bytes, int pal_entries)
{
    (void) mirror;      // the word lists already say which orientations exist
    if (n_masks == 0 || n_targets == 0) return 0;
    if (!occ || !groups || bpitch != occupancy_tile_pitch(g.W)) return 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (!scratch.work_counter || !scratch.acc) return 0;
    cudaMemsetAsync(scratch.work_counter, 0, sizeof(unsigned long long), s);
    cudaMemsetAsync(scratch.acc, 0, kMatchAccBytes, s);
    if (wide_lpal) pal_entries = 0;         // WIDE lists carry their intervals: no palette is staged
    const int warps = cand_launch_shape(xy_shift, g, pal_entries).warps;
    const int staged = cand_staged_palette(pal_entries);
#define CDS_CAND_LAUNCH(NCW) launch_cfg<CDS_PALETTE_GROUP, NCW>(masks, n_masks, planes, g, n_targets, occ, bpitch, groups, xy_shift, scores, scratch, s, dev, wide_lpal, band_bytes, staged)
    if (warps >= 31) return CDS_CAND_LAUNCH(31);
    if (warps >= 28) return CDS_CAND_LAUNCH(28);
    if (warps >= 24) return CDS_CAND_LAUNCH(24);
    return CDS_CAND_LAUNCH(16);
#undef CDS_CAND_LAUNCH
}

}  // namespace cds

// cds_ingest.cu -- device side of the image ingest (SURVEY 8f, row f4): PackBits / stored TIFF strips -> RGB pixels.
//
// Replaces, for targets that arrive as TIFF files, the JVM-side decode of the reference:
// ImageArrayUtils.readImageArrayRangeWithTiffReader + packBitsUncompress
// (colormipsearch-api/src/main/java/org/janelia/colormipsearch/imageprocessing/ImageArrayUtils.java:184-258).
// The host reads only the tags (cds_tiff.cpp); the strips cross PCIe as stored -- colour-depth MIPs are mostly black, so
// PackBits shrinks the 2 MB of a 1210x566 image to 65-255 kB -- and are expanded here, next to the encoder that consumes them.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <thread>

#include "cds_runtime.h"
#include "cds_tiff.h"

using namespace cds;

#define CDS_TRY(expr) do { cds_status _s = (expr); if (_s != CDS_OK) return _s; } while (0)
#define CDS_CUDA(ctx, expr) CDS_TRY((ctx)->check((expr), #expr))

namespace {

constexpr int kDecodeWarps = 8;
constexpr int kDecodeBuf = 2048;       // bytes of decoded output a warp collects in shared memory before it writes them out
constexpr int kDecodeSlack = 128;      // the longest run: a run that starts inside the buffer always fits

// Writes the first `n_buf` bytes of a warp's buffer to global memory.  Buffer byte b is strip byte `first + b` (first may be
// negative: the buffer window is aligned to 16 bytes in GLOBAL memory, so up to 15 bytes in front of the strip's first byte
// and behind its last one belong to the neighbouring strips and must not be touched).  Whole 16-byte vectors inside the strip
// go out as one 128-bit store per lane, fully coalesced; the ragged ends byte by byte.
__device__ __forceinline__ void flush_window(const uint8_t *sb, uint8_t *gout, int first, uint32_t n_buf, uint32_t out_len, uint32_t lane)
{
    __syncwarp();
    for (uint32_t v = lane; v * 16 < n_buf; v += 32) {
        const int lo = first + (int) (v * 16);
        if (lo >= 0 && lo + 16 <= (int) out_len && v * 16 + 16 <= n_buf) {
            *reinterpret_cast<uint4 *>(gout + lo) = *reinterpret_cast<const uint4 *>(sb + v * 16);
        } else {
            for (uint32_t b = 0; b < 16 && v * 16 + b < n_buf; b++) {
                const int o = lo + (int) b;
                if (o >= 0 && o < (int) out_len) gout[o] = sb[v * 16 + b];
            }
        }
    }
    __syncwarp();
}

__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_u8(uint32_t addr, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" :: "r"(addr), "r"(v) : "memory"); }

// One warp per strip.  PackBits is a chain of runs whose positions depend on every control byte before them, so a strip is
// inherently serial in its control bytes -- but a chunk of 1 024 images has ~73 000 strips, enough to keep every SM's warp
// slots full, and a colour-depth MIP is mostly black: of its ~30 000 runs most are 128-byte fills with the same value that
// follow each other.  What counts is the number of instructions per run, so every iteration of the loop below takes as many
// CONSECUTIVE EQUAL-VALUE FILL RUNS as it can see at once: lane i reads the byte pair at input position idx + 2 i, a ballot
// finds how many leading pairs are fill runs of the first pair's value, one warp reduction adds their lengths, and the
// whole stretch (a black image row is 29 runs) is written as a single fill.  Literal runs are copied 32 bytes per step.
// Output is collected in a per-warp shared-memory window aligned with global memory and leaves the SM as full 128-bit
// stores (byte stores straight to global memory made every run a handful of partial-sector writes).
// (A lane-per-strip variant, one run state machine per lane, was 2.4 x slower: a third of all 4-byte output words contain
// a run boundary of SOME lane, so the warp lived in the divergent slow path with ~8 of 32 lanes active.)
// Like the reference's loop (ImageArrayUtils.java:229-258): 0..127 = that many + 1 literal bytes, -127..-1 = repeat the next
// byte 1 - n times, -128 = no-op; decoding stops at the end of the strip's input or of its rows, and whatever was not
// produced stays 0 (the Java array is zero-initialised).  Stored (uncompressed) pieces take the literal path.
__global__ void __launch_bounds__(kDecodeWarps * 32)
tiff_decode_kernel(const uint8_t *__restrict__ src, const TiffStrip *__restrict__ strips, int64_t n_strips, uint8_t *__restrict__ dst)
{
    __shared__ __align__(16) uint8_t s_buf[kDecodeWarps][kDecodeBuf + kDecodeSlack];
    const uint32_t lane = threadIdx.x & 31;
    const int64_t w = (int64_t) blockIdx.x * kDecodeWarps + (threadIdx.x >> 5);
    if (w >= n_strips) return;
    uint8_t *sb = s_buf[threadIdx.x >> 5];
    const uint32_t sba = (uint32_t) __cvta_generic_to_shared(sb);
    const TiffStrip st = strips[w];
    const uint8_t *__restrict__ in = src + st.src;
    const uint32_t in_len = st.src_len, out_len = st.dst_len & ~kTiffStripPacked;
    const bool packed = (st.dst_len & kTiffStripPacked) != 0;
    uint8_t *gout = dst + st.dst;
    const uint32_t mis = (uint32_t) (reinterpret_cast<uintptr_t>(gout) & 15);     // the window starts at the 16-byte boundary below gout

    uint32_t pos = 0, idx = 0;         // strip-relative output / input positions
    uint32_t flushed = 0;              // window bytes already written out (a multiple of kDecodeBuf)
    while (pos < out_len) {
        uint32_t cnt, fill = 0, from = 0;
        bool copy = false;
        if (idx >= in_len) {
            cnt = out_len - pos;                                   // input used up: zeros to the end of the strip
        } else if (!packed) {
            cnt = min((uint32_t) kDecodeSlack, in_len - idx);
            copy = true; from = idx; idx += cnt;
        } else {
            // lane i looks at the pair (control, value) that starts at idx + 2 i
            const uint32_t q = idx + 2 * lane;
            const uint32_t c = q < in_len ? (uint32_t) in[q] : 0u;
            const uint32_t v = q + 1 < in_len ? (uint32_t) in[q + 1] : 0u;
            const uint32_t c0 = __shfl_sync(0xffffffffu, c, 0), v0 = __shfl_sync(0xffffffffu, v, 0);
            if (c0 < 128) { cnt = c0 + 1; copy = true; from = idx + 1; idx += 1 + cnt; }
            else if (c0 == 128) { idx += 1; continue; }
            else {
                const uint32_t same = __ballot_sync(0xffffffffu, c > 128 && v == v0 && q + 1 < in_len);
                const uint32_t k = same == 0xffffffffu ? 32u : (uint32_t) __ffs((int) ~same) - 1u;      // >= 1 unless the value byte is missing
                fill = v0;
                if (k == 0) { cnt = 257 - c0; fill = 0; idx += 2; }                                       // a fill whose value byte lies beyond the input
                else { cnt = __reduce_add_sync(0xffffffffu, lane < k ? 257 - c : 0u); idx += 2 * k; }
            }
        }
        uint32_t todo = min(cnt, out_len - pos);
        if (copy) {
            // a literal of at most 128 bytes: it fits behind any position inside the buffer
            const uint32_t bi = pos + mis - flushed;
            for (uint32_t i = lane; i < todo; i += 32) sts_u8(sba + bi + i, from + i < in_len ? (uint32_t) in[from + i] : 0u);
            pos += todo;
            todo = 0;
        }
        const uint32_t vw = fill * 0x01010101u;
        for (;;) {
            // a fill of `todo` bytes, as much as the buffer takes: aligned words [a, e), head bytes [bi, 4a), tail bytes [4e, end)
            if (todo) {
                const uint32_t bi = pos + mis - flushed;
                const uint32_t n = min(todo, (uint32_t) (kDecodeBuf + kDecodeSlack) - bi);
                const uint32_t a = (bi + 3) >> 2, e = (bi + n) >> 2;
                if (a < e) {
                    for (uint32_t x = a + lane; x < e; x += 32) sts_u32(sba + 4 * x, vw);
                    if (lane < 4 * a - bi) sts_u8(sba + bi + lane, fill);
                    if (lane < bi + n - 4 * e) sts_u8(sba + 4 * e + lane, fill);
                } else if (lane < n) {
                    sts_u8(sba + bi + lane, fill);
                }
                pos += n; todo -= n;
            }
            if (pos + mis - flushed < (uint32_t) kDecodeBuf) break;
            flush_window(sb, gout, (int) flushed - (int) mis, kDecodeBuf, out_len, lane);
            // carry the bytes beyond the window (at most kDecodeSlack) to its start
            const uint32_t over = pos + mis - flushed - kDecodeBuf;
            const uint32_t wv = lane * 4 < over ? *reinterpret_cast<const uint32_t *>(sb + kDecodeBuf + lane * 4) : 0u;
            __syncwarp();
            if (lane * 4 < over) *reinterpret_cast<uint32_t *>(sb + lane * 4) = wv;
            __syncwarp();              // the carried words may reach past `over`, where the next run writes
            flushed += kDecodeBuf;
        }
    }
    flush_window(sb, gout, (int) flushed - (int) mis, pos + mis - flushed, out_len, lane);
}

}  // namespace

namespace {
// ------------------------------------------------------------------------------------------------------------------
// Fused ingest: PackBits / stored strips -> the library's code words and per-sector "can match" bits, with no RGB image in HBM in
// between (the streaming search's chunks used to be decoded to RGB, written out, and read back by encode_rgb_kernel).
//
// One warp per strip again -- PackBits is serial in its control bytes -- but the warp owns ONE IMAGE ROW of decoded bytes in
// shared memory instead of a window of the output image.  A colour-depth MIP is mostly black, and a black stretch is a chain of
// zero fills: those only advance the output position (the row buffer starts out, and is left, all zero).  Literal runs and
// non-zero fills are written into the row buffer and mark the 32-pixel chunks they touch.  When the position passes the end of
// the row the row is emitted: the whole row of code words is written as the black code word with 128-bit stores (pad columns
// included), then only the marked chunks are looked at -- their non-black pixels are compacted into a small queue so that the
// colour classifier (~150 instructions) runs on full warps, and their code words and sector bits patch the row.  Work is
// proportional to the image's content, not to its area.  Same decoding rules as tiff_decode_kernel (and the reference's
// packBitsUncompress, ImageArrayUtils.java:229-258): decoding stops at the end of the strip's input or of its rows, whatever was
// not produced stays black.
__device__ __forceinline__ int fuse_classify(int r, int g, int b, int &second, int &maxv)
{
    if (b > r && b > g) { maxv = b; if (r > g) { second = r; return 0; } second = g; return 1; }
    if (g > b && g > r) { maxv = g; if (b > r) { second = b; return 2; } second = r; return 3; }
    if (r > b && r > g) { maxv = r; if (g > b) { second = g; return 4; } second = b; return 5; }
    maxv = max(r, max(g, b));
    second = 0;
    return -1;
}

// the code word of cds_common.h (the same arithmetic as encode_color_dev in cds_kernels.cu; test_encode_all_16M_colours pins both
// through searches over files == searches over pixels)
__device__ __forceinline__ uint32_t fuse_encode(int r, int g, int b, const uint16_t *__restrict__ rank_tab, int thr, int &sector)
{
    int second, maxv;
    sector = fuse_classify(r, g, b, second, maxv);
    const uint32_t sr = sector < 0 ? (uint32_t) CDS_SR_NONE : (uint32_t) sector * CDS_SECTOR_STRIDE + __ldg(rank_tab + second * 256 + maxv);
    uint32_t code = (sr << CDS_CODE_SR_SHIFT) | (uint32_t) maxv;
    if (!(maxv > thr)) { code |= CDS_CODE_BELOW_BIT; sector = -1; }
    return code;
}

constexpr int kFuseWarps = 8;
constexpr int kFuseQueue = 64;

// One strip, by one warp (below: warps fetch strips from a counter until none is left -- strips differ a lot in cost, and a CTA of eight
// warps that each took exactly one strip kept its registers and shared memory until its slowest warp was done: 34 % achieved occupancy).
__device__ __forceinline__ void tiff_encode_strip(const int64_t w, const uint32_t lane, const uint32_t warp, uint4 *s_fuse4,
                                                  const uint8_t *__restrict__ src, const TiffStrip *__restrict__ strips, uint32_t *__restrict__ planes,
                                                  const PlaneGeom &g, int64_t first_slot, const uint16_t *__restrict__ rank_tab, int thr, int vp,
                                                  uint32_t *__restrict__ valid, int row_buf_bytes)
{
    const int valid_words = CDS_NUM_SECTORS * vp;
    const int per_warp = row_buf_bytes + valid_words * 4 + kFuseQueue * 4;           // multiples of 16
    uint8_t *rowbuf = reinterpret_cast<uint8_t *>(s_fuse4) + (size_t) warp * per_warp;
    uint32_t *s_valid = reinterpret_cast<uint32_t *>(rowbuf + row_buf_bytes);
    uint32_t *s_queue = s_valid + valid_words;
    const uint32_t rowbuf_a = (uint32_t) __cvta_generic_to_shared(rowbuf);

    const TiffStrip st = strips[w];
    const uint8_t *__restrict__ in = src + st.src;
    const uint32_t in_len = st.src_len, out_len = st.dst_len & ~kTiffStripPacked;
    const bool packed = (st.dst_len & kTiffStripPacked) != 0;
    const uint32_t row_bytes = (uint32_t) g.W * 3u;
    const int64_t img = st.dst / (uint32_t) g.H;                                      // strips and stored pieces are whole rows: dst counts rows
    int y = (int) (st.dst % (uint32_t) g.H);
    const int y_end = y + (int) (out_len / row_bytes);
    const uint32_t black = (uint32_t) CDS_SR_NONE << CDS_CODE_SR_SHIFT | (0 > thr ? 0u : CDS_CODE_BELOW_BIT);

    for (int k = lane; k < (row_buf_bytes + valid_words * 4) / 16; k += 32) reinterpret_cast<uint4 *>(rowbuf)[k] = make_uint4(0u, 0u, 0u, 0u);
    __syncwarp();

    uint32_t dirty_lo = 0, dirty_hi = 0;           // 32-pixel chunks of the current row that hold decoded non-zero bytes (uniform)
    uint32_t row_start = 0;                        // strip-relative output position of the current row's first byte
    const uint32_t lt = (1u << lane) - 1u;

    // The decoder.  PackBits is a chain of runs, but the chain can be followed 32 input bytes at a time: every lane takes one byte
    // of the window, works out where the NEXT control byte would be if its byte were one, pointer doubling (four shuffles) and five
    // OR-reductions mark the bytes that really are control bytes, and a warp scan over the runs' lengths gives every run its place
    // in the output.  Zero fills -- most runs of a mostly black image -- then cost nothing more; literal bytes that lie inside the
    // window are stored by the lanes that hold them, in one step for all literal runs of the window; non-zero fills and the tail
    // of a literal that leaves the window are short cooperative loops.  (The first version took one run, or one stretch of equal
    // fills, per iteration: ~16 500 iterations of ~130 instructions per image, profiles/r02_fuse_v1_ncu_summary.txt.)
    // A window whose writes would cross the end of the current row falls back to a generic one-run-at-a-time step (`span`), which
    // also serves stored strips.  One loop with one site per step: the steps are long, several inlined copies would not fit the
    // instruction cache.
    uint32_t pos = 0, idx = 0;
    uint32_t span_a = 0, span_n = 0, span_from = 0, span_fill = 0;     // generic step: decoded bytes [span_a, span_a + span_n) still to write
    bool span_lit = false;
    uint32_t emit_to = 0;                          // rows that end at or before this position are complete: emit them before the next write
    bool done = false;
    for (;;) {
        const uint32_t row_end = row_start + row_bytes;
        if (done ? y < y_end : row_end <= emit_to) {
            // ------------------------------------------------------------------ emit the current row
            uint32_t *drow = planes + g.row_offset(first_slot + img, y);
            // the whole row black, pad columns as pad words (the row is 16-byte aligned and a multiple of four words long)
            for (int v4 = (int) lane; v4 < g.pitch / 4; v4 += 32) {
                const int x = 4 * v4;
                uint4 w4 = make_uint4(black, black, black, black);
                if (x + 3 >= g.W) {                            // the one or two words where the image ends
                    w4.x = x < g.W ? black : CDS_CODE_PAD_WORD; w4.y = x + 1 < g.W ? black : CDS_CODE_PAD_WORD;
                    w4.z = x + 2 < g.W ? black : CDS_CODE_PAD_WORD; w4.w = CDS_CODE_PAD_WORD;
                }
                reinterpret_cast<uint4 *>(drow)[v4] = w4;
            }
            const bool dirty = (dirty_lo | dirty_hi) != 0u;
            if (dirty) {
                __syncwarp();                  // the black words above are ordered before the patches below
                // non-black pixels of the marked chunks -> queue -> colour classifier on full warps
                uint32_t qh = 0, qt = 0;
                uint32_t m = dirty_lo;
                int cbase = 0;
                for (;;) {
                    bool more = true;
                    if (m == 0u) {
                        if (cbase == 0) { m = dirty_hi; cbase = 32; }
                        if (m == 0u) more = false;
                    }
                    if (more) {
                        const int c = (__ffs((int) m) - 1) + cbase;
                        m &= m - 1;
                        const int x = 32 * c + (int) lane;
                        bool lit = false;
                        if (x < g.W) lit = (rowbuf[3 * x] | rowbuf[3 * x + 1] | rowbuf[3 * x + 2]) != 0;
                        const unsigned bal = __ballot_sync(0xffffffffu, lit);
                        if (lit) s_queue[(qt + (uint32_t) __popc(bal & lt)) & (kFuseQueue - 1)] = (uint32_t) x;
                        qt += (uint32_t) __popc(bal);
                        __syncwarp();
                    }
                    // classify when 32 pixels wait (or, after the last chunk, whatever is left)
                    while (qt - qh >= 32u || (!more && qt != qh)) {
                        const uint32_t nq = min(32u, qt - qh);
                        if (lane < nq) {
                            const int x = (int) s_queue[(qh + lane) & (kFuseQueue - 1)];
                            const uint8_t *px = rowbuf + 3 * x;
                            int sector;
                            const uint32_t code = fuse_encode(px[0], px[1], px[2], rank_tab, thr, sector);
                            drow[x] = code;
                            if (valid && sector >= 0) atomicOr(&s_valid[sector * vp + (x >> 5)], 1u << (x & 31));
                        }
                        qh += nq;
                        __syncwarp();
                    }
                    if (!more) break;
                }
            }
            if (valid) {
                uint4 *vout = reinterpret_cast<uint4 *>(valid + ((size_t) img * g.H + y) * valid_words);
                for (int k = (int) lane; k < valid_words / 4; k += 32) vout[k] = reinterpret_cast<const uint4 *>(s_valid)[k];
            }
            if (dirty) {
                __syncwarp();
                for (int k = (int) lane; k < (row_buf_bytes + valid_words * 4) / 16; k += 32) reinterpret_cast<uint4 *>(rowbuf)[k] = make_uint4(0u, 0u, 0u, 0u);
                __syncwarp();
            }
            dirty_lo = dirty_hi = 0u;
            y++;
            row_start += row_bytes;
            continue;
        }
        if (done) break;
        if (span_n) {
            // ---------------------------------------------------------------------- generic step: the piece of the span inside this row
            if (span_a >= row_end) { emit_to = span_a; continue; }
            const uint32_t off = span_a - row_start;
            const uint32_t take = min(span_n, row_bytes - off);
            for (uint32_t i = lane; i < take; i += 32) {
                uint32_t b = span_fill;
                if (span_lit) b = span_from + i < in_len ? (uint32_t) in[span_from + i] : 0u;
                asm volatile("st.shared.u8 [%0], %1;" :: "r"(rowbuf_a + off + i), "r"(b) : "memory");
            }
            const uint32_t c0 = off / 96u, c1 = (off + take - 1u) / 96u;                 // chunk = 32 pixels = 96 bytes
            for (uint32_t c = c0; c <= c1; c++) { if (c < 32u) dirty_lo |= 1u << c; else dirty_hi |= 1u << (c - 32u); }
            span_a += take; span_n -= take; span_from += take;
            __syncwarp();
            continue;
        }
        if (!(pos < out_len && idx < in_len)) { done = true; continue; }
        if (!packed) {
            span_n = min(min(in_len - idx, out_len - pos), 4096u);
            span_a = pos; span_lit = true; span_from = idx;
            pos += span_n; idx += span_n;
            continue;
        }
        // -------------------------------------------------------------------------- a window of 32 input bytes
        const uint32_t p = idx + lane;
        const uint32_t c = p < in_len ? (uint32_t) in[p] : 128u;
        uint32_t v = __shfl_down_sync(0xffffffffu, c, 1);
        const bool v_missing = p + 1 >= in_len;                        // a fill whose value byte lies beyond the input fills with 0
        if (v_missing) v = 0u;
        const bool is_lit = c < 128u, is_fill = c > 128u;
        const uint32_t consumed = is_lit ? c + 2u : (is_fill ? 2u : 1u);
        const uint32_t len = is_lit ? c + 1u : (is_fill ? 257u - c : 0u);
        // a control byte can be taken in this window when its header is here: a fill needs its value byte (lane 31 only has it when the input ends)
        const bool takeable = p < in_len && (!is_fill || lane < 31u || v_missing);
        const uint32_t nxt = lane + consumed;
        uint32_t j1 = (takeable && nxt < 32u && idx + nxt < in_len) ? nxt : 32u;     // 32 = the chain leaves the window
        uint32_t t2 = __shfl_sync(0xffffffffu, j1, (int) (j1 & 31u));
        const uint32_t j2 = j1 < 32u ? t2 : 32u;
        t2 = __shfl_sync(0xffffffffu, j2, (int) (j2 & 31u));
        const uint32_t j4 = j2 < 32u ? t2 : 32u;
        t2 = __shfl_sync(0xffffffffu, j4, (int) (j4 & 31u));
        const uint32_t j8 = j4 < 32u ? t2 : 32u;
        t2 = __shfl_sync(0xffffffffu, j8, (int) (j8 & 31u));
        const uint32_t j16 = j8 < 32u ? t2 : 32u;
        uint32_t T = 1u;                                               // the control bytes of the window: byte 0 and everything the chain reaches
        T |= __reduce_or_sync(0xffffffffu, ((T >> lane) & 1u) && j16 < 32u ? 1u << j16 : 0u);
        T |= __reduce_or_sync(0xffffffffu, ((T >> lane) & 1u) && j8 < 32u ? 1u << j8 : 0u);
        T |= __reduce_or_sync(0xffffffffu, ((T >> lane) & 1u) && j4 < 32u ? 1u << j4 : 0u);
        T |= __reduce_or_sync(0xffffffffu, ((T >> lane) & 1u) && j2 < 32u ? 1u << j2 : 0u);
        T |= __reduce_or_sync(0xffffffffu, ((T >> lane) & 1u) && j1 < 32u ? 1u << j1 : 0u);
        const bool run = ((T >> lane) & 1u) && takeable;               // this lane's byte starts a run that this window decodes
        // (the last control byte of the chain may be a fill cut off by the window's end: it starts the next window)
        const uint32_t last = 31u - (uint32_t) __clz((int) T);
        const bool last_taken = __shfl_sync(0xffffffffu, (int) takeable, (int) last) != 0;
        const uint32_t last_next = __shfl_sync(0xffffffffu, nxt, (int) last);
        const uint32_t new_idx = idx + (last_taken ? last_next : last);
        // where every run starts in the output
        const uint32_t mylen = run ? len : 0u;
        uint32_t incl = mylen;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int) lane >= d) incl += u;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        const uint32_t start = pos + incl - mylen;
        const bool writes = run && start < out_len && (is_lit || (is_fill && v != 0u));
        const uint32_t wend = min(start + len, out_len);
        const uint32_t w_min = __reduce_min_sync(0xffffffffu, writes ? start : 0xffffffffu);
        if (w_min == 0xffffffffu) { pos += total; idx = new_idx; continue; }          // nothing but zero fills and no-ops
        if (w_min >= row_end) { emit_to = w_min; continue; }                           // finish the rows in between, then look at this window again
        const uint32_t w_max = __reduce_max_sync(0xffffffffu, writes ? wend : 0u);
        if (w_max > row_end) {
            // the window's writes cross the end of the row: take its first run alone, generically
            const uint32_t c0 = __shfl_sync(0xffffffffu, c, 0), v0 = __shfl_sync(0xffffffffu, v, 0);
            const uint32_t len0 = c0 < 128u ? c0 + 1u : (c0 > 128u ? 257u - c0 : 0u);
            span_a = pos; span_lit = c0 < 128u; span_from = idx + 1u; span_fill = v0;
            span_n = (c0 < 128u || (c0 > 128u && v0 != 0u)) ? min(len0, out_len - pos) : 0u;
            pos += len0;
            idx += c0 < 128u ? c0 + 2u : (c0 > 128u ? 2u : 1u);
            continue;
        }
        // ------------------------------------------------------------------------------ all writes of the window land in the current row
        const uint32_t base = rowbuf_a - row_start;                    // row buffer address of output position 0 (wraps; only sums are used)
        uint32_t d_lo = 0u, d_hi = 0u;
        // literal bytes inside the window: the lane that holds the byte stores it
        const uint32_t lit_runs = __ballot_sync(0xffffffffu, run && is_lit);
        {
            const uint32_t below = lit_runs & lt;
            const int owner = below ? 31 - __clz((int) below) : 0;
            const uint32_t oc = __shfl_sync(0xffffffffu, c, owner), ostart = __shfl_sync(0xffffffffu, start, owner);
            const uint32_t d = lane - (uint32_t) owner - 1u;
            if (below && d <= oc) {
                const uint32_t o = ostart + d;
                if (o < out_len) {
                    const uint32_t b = p < in_len ? c : 0u;
                    asm volatile("st.shared.u8 [%0], %1;" :: "r"(base + o), "r"(b) : "memory");
                    const uint32_t ch = (o - row_start) / 96u;
                    if (ch < 32u) d_lo |= 1u << ch; else d_hi |= 1u << (ch - 32u);
                }
            }
        }
        // the tail of a literal that leaves the window (only the last run can)
        if (last_taken && last_next > 32u && ((lit_runs >> last) & 1u)) {
            const uint32_t lstart = __shfl_sync(0xffffffffu, start, (int) last);
            const uint32_t done_bytes = 31u - last;                    // data bytes of the run that were inside the window
            const uint32_t extra = last_next - 32u;
            for (uint32_t e = lane; e < extra; e += 32) {
                const uint32_t o = lstart + done_bytes + e;
                if (o < out_len) {
                    const uint32_t src_i = idx + 32u + e;
                    const uint32_t b = src_i < in_len ? (uint32_t) in[src_i] : 0u;
                    asm volatile("st.shared.u8 [%0], %1;" :: "r"(base + o), "r"(b) : "memory");
                    const uint32_t ch = (o - row_start) / 96u;
                    if (ch < 32u) d_lo |= 1u << ch; else d_hi |= 1u << (ch - 32u);
                }
            }
        }
        // non-zero fills, one after the other
        uint32_t fills = __ballot_sync(0xffffffffu, writes && is_fill);
        while (fills) {
            const int f = __ffs((int) fills) - 1;
            fills &= fills - 1;
            const uint32_t fs = __shfl_sync(0xffffffffu, start, f), fe = __shfl_sync(0xffffffffu, wend, f), fv = __shfl_sync(0xffffffffu, v, f);
            for (uint32_t o = fs + lane; o < fe; o += 32) {
                asm volatile("st.shared.u8 [%0], %1;" :: "r"(base + o), "r"(fv) : "memory");
                const uint32_t ch = (o - row_start) / 96u;
                if (ch < 32u) d_lo |= 1u << ch; else d_hi |= 1u << (ch - 32u);
            }
        }
        dirty_lo |= __reduce_or_sync(0xffffffffu, d_lo);
        dirty_hi |= __reduce_or_sync(0xffffffffu, d_hi);
        pos += total;
        idx = new_idx;
        __syncwarp();
    }
}

__global__ void __launch_bounds__(kFuseWarps * 32)
tiff_encode_kernel(const uint8_t *__restrict__ src, const TiffStrip *__restrict__ strips, int64_t n_strips, uint32_t *__restrict__ planes,
                   PlaneGeom g, int64_t first_slot, const uint16_t *__restrict__ rank_tab, int thr, int vp,
                   uint32_t *__restrict__ valid /* chunk-relative [n][H][sectors][vp], or nullptr */, int row_buf_bytes,
                   unsigned long long *__restrict__ next_strip /* zero on entry */)
{
    extern __shared__ uint4 s_fuse4[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (;;) {
        unsigned long long w = 0;
        if (lane == 0) w = atomicAdd(next_strip, 1ull);
        w = __shfl_sync(0xffffffffu, w, 0);
        if (w >= (unsigned long long) n_strips) return;
        tiff_encode_strip((int64_t) w, lane, warp, s_fuse4, src, strips, planes, g, first_slot, rank_tab, thr, vp, valid, row_buf_bytes);
        __syncwarp();
    }
}

}  // namespace

void cds::launch_tiff_encode(const uint8_t *src, const TiffStrip *strips, int64_t n_strips, uint32_t *planes, PlaneGeom g, int64_t first_slot,
                             const uint16_t *rank_tab, int data_threshold, uint32_t *valid, unsigned long long *work_counter, cudaStream_t s)
{
    if (n_strips <= 0) return;
    const int vp = occupancy_valid_pitch(g.W);
    const int row_buf = (g.W * 3 + 15) / 16 * 16;
    const size_t smem = (size_t) kFuseWarps * (row_buf + CDS_NUM_SECTORS * vp * 4 + kFuseQueue * 4);
    static bool attr_set = false;
    if (!attr_set) { cudaFuncSetAttribute(tiff_encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); attr_set = true; }
    // a persistent grid: as many CTAs as fit the device at once, every warp takes strips until the counter runs out
    static int resident_blocks = 0;
    if (resident_blocks == 0) {
        int per_sm = 0, dev = 0, n_sm = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tiff_encode_kernel, kFuseWarps * 32, smem);
        resident_blocks = std::max(1, per_sm) * n_sm;
    }
    const int64_t blocks = std::min<int64_t>((n_strips + kFuseWarps - 1) / kFuseWarps, resident_blocks);
    cudaMemsetAsync(work_counter, 0, sizeof(unsigned long long), s);
    tiff_encode_kernel<<<(unsigned) blocks, kFuseWarps * 32, smem, s>>>(src, strips, n_strips, planes, g, first_slot, rank_tab, data_threshold, vp, valid, row_buf,
                                                                        work_counter);
}

void cds::launch_tiff_decode(const uint8_t *src, const TiffStrip *strips, int64_t n_strips, uint8_t *dst_rgb, cudaStream_t s)
{
    if (n_strips <= 0) return;
    const int64_t blocks = (n_strips + kDecodeWarps - 1) / kDecodeWarps;
    tiff_decode_kernel<<<(unsigned) blocks, kDecodeWarps * 32, 0, s>>>(src, strips, n_strips, dst_rgb);
}

namespace {

// Strip table of files [i0, i0 + cnt): sources relative to the first byte of file i0, destinations relative to image i0.
cds_status collect_chunk(cds_ctx *ctx, const char *who, const uint8_t *blob, const int64_t *offsets, int64_t i0, int64_t cnt,
                         int W, int H, std::vector<TiffStrip> &strips)
{
    strips.clear();
    const size_t img_bytes = (size_t) W * H * 3;
    const int64_t base = offsets[i0];
    std::string err;
    for (int64_t i = 0; i < cnt; i++) {
        const int64_t a = offsets[i0 + i], b = offsets[i0 + i + 1];
        if (a < 0 || b < a) return ctx->fail(CDS_ERR_BAD_ARG, std::string(who) + ": offsets must be non-decreasing");
        cds_status s = tiff_collect_strips(blob + a, (size_t) (b - a), W, H, (uint64_t) (a - base), (uint64_t) i * img_bytes, strips, err);
        if (s != CDS_OK) return ctx->fail(s, std::string(who) + ": file " + std::to_string(i0 + i) + ": " + err);
    }
    return CDS_OK;
}

}  // namespace

namespace cds {

// Uploads files [i0, i0 + cnt) and decodes them into d_rgb, everything on stream `s` (used by the library and the one-shot
// decoder; the streaming search has its own double-buffered version).  d_comp / d_strips must hold the chunk.
cds_status ingest_chunk(cds_ctx *ctx, const char *who, const uint8_t *blob, const int64_t *offsets, int64_t i0, int64_t cnt, int W, int H,
                        uint8_t *d_comp, size_t comp_cap, TiffStrip *d_strips, size_t strips_cap, uint8_t *d_rgb, cudaStream_t s,
                        std::vector<TiffStrip> &strips)
{
    CDS_TRY(collect_chunk(ctx, who, blob, offsets, i0, cnt, W, H, strips));
    const size_t bytes = (size_t) (offsets[i0 + cnt] - offsets[i0]);
    if (bytes > comp_cap || strips.size() > strips_cap) return ctx->fail(CDS_ERR_CAPACITY, std::string(who) + ": internal staging too small");
    CDS_CUDA(ctx, cudaMemcpyAsync(d_comp, blob + offsets[i0], bytes, cudaMemcpyHostToDevice, s));
    // the table is pageable host memory: the runtime stages it before the call returns, so `strips` may be reused
    CDS_CUDA(ctx, cudaMemcpyAsync(d_strips, strips.data(), strips.size() * sizeof(TiffStrip), cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += (int64_t) bytes + (int64_t) (strips.size() * sizeof(TiffStrip));
    launch_tiff_decode(d_comp, d_strips, (int64_t) strips.size(), d_rgb, s);
    ctx->stats.kernel_launches++;
    CDS_CUDA(ctx, cudaGetLastError());
    return CDS_OK;
}

// upper bounds for the staging of up to `cnt` consecutive files of the blob
void ingest_bounds(const int64_t *offsets, int64_t n, int64_t cnt, int W, int H, size_t &comp_cap, size_t &strips_cap)
{
    int64_t worst = 0;
    for (int64_t i = 0; i < n; i += cnt) worst = std::max(worst, offsets[std::min(n, i + cnt)] - offsets[i]);
    comp_cap = (size_t) std::max<int64_t>(worst, 0) + 64;
    strips_cap = (size_t) cnt * tiff_strips_bound(W, H);
}

}  // namespace cds

extern "C" cds_status cds_tiff_decode_rgb(cds_ctx *ctx, const uint8_t *blob, const int64_t *offsets, int64_t n,
                                          int32_t width, int32_t height, uint8_t *out_rgb)
{
    return cds::abi_guard("cds_tiff_decode_rgb", [&]() -> cds_status {
        if (!ctx) { set_tls_error("cds_tiff_decode_rgb: NULL context"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (n < 0 || width <= 0 || height <= 0 || width > 16384 || height > 16384) return ctx->fail(CDS_ERR_BAD_ARG, "cds_tiff_decode_rgb: bad size");
        if (n == 0) return CDS_OK;
        if (!blob || !offsets || !out_rgb) return ctx->fail(CDS_ERR_BAD_ARG, "cds_tiff_decode_rgb: NULL argument");
        DevState &ds = ctx->devs[0];
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        const size_t img_bytes = (size_t) width * height * 3;
        const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(64, (int64_t) ((size_t) 1 << 30) / (int64_t) img_bytes));
        size_t comp_cap, strips_cap;
        ingest_bounds(offsets, n, chunk, width, height, comp_cap, strips_cap);
        uint8_t *d_comp = nullptr, *d_rgb = nullptr;
        TiffStrip *d_strips = nullptr;
        auto release = [&]() { cudaStreamSynchronize(ds.stream); ds.pool.free(d_comp); ds.pool.free(d_rgb); ds.pool.free(d_strips); };
        struct Guard { std::function<void()> f; ~Guard() { f(); } } guard{release};
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_comp, comp_cap));
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_strips, strips_cap * sizeof(TiffStrip)));
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_rgb, (size_t) chunk * img_bytes));
        std::vector<TiffStrip> strips;
        for (int64_t i0 = 0; i0 < n; i0 += chunk) {
            const int64_t cnt = std::min(chunk, n - i0);
            CDS_TRY(ingest_chunk(ctx, "cds_tiff_decode_rgb", blob, offsets, i0, cnt, width, height, d_comp, comp_cap, d_strips, strips_cap, d_rgb, ds.stream, strips));
            CDS_CUDA(ctx, cudaMemcpyAsync(out_rgb + (size_t) i0 * img_bytes, d_rgb, (size_t) cnt * img_bytes, cudaMemcpyDeviceToHost, ds.stream));
            CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
            ctx->stats.d2h_bytes += (int64_t) cnt * (int64_t) img_bytes;
        }
        return CDS_OK;
    });
}

extern "C" cds_status cds_library_add_tiff(cds_library *lib, const uint8_t *blob, const int64_t *offsets, int64_t n, int64_t *first_index)
{
    return cds::abi_guard("cds_library_add_tiff", [&]() -> cds_status {
        if (!lib) { set_tls_error("cds_library_add_tiff: NULL library"); return CDS_ERR_BAD_ARG; }
        cds_ctx *ctx = lib->ctx;
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (n < 0) return ctx->fail(CDS_ERR_BAD_ARG, "negative image count");
        if (n > 0 && (!blob || !offsets)) return ctx->fail(CDS_ERR_BAD_ARG, "cds_library_add_tiff: NULL argument");
        if (n == 0) return library_append(lib, 0, nullptr, first_index);
        const int W = lib->g.W, H = lib->g.H;
        // library_append hands out runs of at most kLibBlock images; bound the staging by any kLibBlock consecutive files
        size_t comp_cap = 0, strips_cap = 0;
        {
            int64_t worst = 0;
            for (int64_t i = 0; i < n; i++) worst = std::max(worst, offsets[std::min(n, i + kLibBlock)] - offsets[i]);
            comp_cap = (size_t) std::max<int64_t>(worst, 0) + 64;
            strips_cap = (size_t) kLibBlock * tiff_strips_bound(W, H);
        }
        const size_t D = ctx->devs.size();
        std::vector<uint8_t *> d_comp(D, nullptr);
        std::vector<TiffStrip *> d_strips(D, nullptr);
        auto release = [&]() {
            for (size_t d = 0; d < D; d++) {
                if (!d_comp[d] && !d_strips[d]) continue;
                cudaSetDevice(ctx->devs[d].dev);
                cudaStreamSynchronize(ctx->devs[d].stream);
                ctx->devs[d].pool.free(d_comp[d]);
                ctx->devs[d].pool.free(d_strips[d]);
            }
        };
        struct Guard { std::function<void()> f; ~Guard() { f(); } } guard{release};
        std::vector<TiffStrip> strips;
        return library_append(lib, n, [&](DevState &ds, int64_t i0, int64_t cnt, uint8_t *d_rgb) -> cds_status {
            const size_t d = (size_t) (&ds - ctx->devs.data());
            if (!d_comp[d]) {
                CDS_CUDA(ctx, ds.pool.alloc((void **) &d_comp[d], comp_cap));
                CDS_CUDA(ctx, ds.pool.alloc((void **) &d_strips[d], strips_cap * sizeof(TiffStrip)));
            }
            return ingest_chunk(ctx, "cds_library_add_tiff", blob, offsets, i0, cnt, W, H, d_comp[d], comp_cap, d_strips[d], strips_cap, d_rgb, ds.stream, strips);
        }, first_index);
    });
}

extern "C" cds_status cds_maskset_add_tiff(cds_maskset *ms, const uint8_t *blob, const int64_t *offsets, int32_t n, int32_t *mask_size_out)
{
    return cds::abi_guard("cds_maskset_add_tiff", [&]() -> cds_status {
        if (!ms) { set_tls_error("cds_maskset_add_tiff: NULL mask set"); return CDS_ERR_BAD_ARG; }
        cds_ctx *ctx = ms->ctx;
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (n < 0 || (n > 0 && (!blob || !offsets))) return ctx->fail(CDS_ERR_BAD_ARG, "cds_maskset_add_tiff: bad arguments");
        if (n == 0) return CDS_OK;
        const int W = ms->W, H = ms->H;
        // maskset_append asks for runs of at most `chunk` masks; uploads and decodes are ordered on one stream, so one buffer does
        const int64_t chunk = maskset_append_chunk(n);
        size_t comp_cap = 0, strips_cap = 0;
        ingest_bounds(offsets, n, chunk, W, H, comp_cap, strips_cap);
        for (int64_t i = 0; i < n; i++) comp_cap = std::max(comp_cap, (size_t) std::max<int64_t>(offsets[std::min<int64_t>(n, i + chunk)] - offsets[i], 0) + 64);
        DevState &d0 = ctx->devs[0];
        CDS_CUDA(ctx, cudaSetDevice(d0.dev));
        // Two sets of upload buffers and a stream of their own for the copies: the files of chunk i + 1 cross PCIe while chunk i is
        // being decoded (maskset_append asks for the chunks in order, one ahead of the preparation kernels).
        uint8_t *d_comp[2] = {nullptr, nullptr};
        TiffStrip *d_strips[2] = {nullptr, nullptr};
        cudaStream_t h2d = nullptr;
        cudaEvent_t up[2] = {nullptr, nullptr}, decoded[2] = {nullptr, nullptr};
        auto release = [&]() {
            if (h2d) cudaStreamSynchronize(h2d);
            cudaStreamSynchronize(d0.copy_stream); cudaStreamSynchronize(d0.stream);
            for (int i = 0; i < 2; i++) {
                d0.pool.free(d_comp[i]); d0.pool.free(d_strips[i]);
                if (up[i]) cudaEventDestroy(up[i]);
                if (decoded[i]) cudaEventDestroy(decoded[i]);
            }
            if (h2d) cudaStreamDestroy(h2d);
        };
        struct Guard { std::function<void()> f; ~Guard() { f(); } } guard{release};
        CDS_CUDA(ctx, cudaStreamCreateWithFlags(&h2d, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CDS_CUDA(ctx, d0.pool.alloc((void **) &d_comp[i], comp_cap));
            CDS_CUDA(ctx, d0.pool.alloc((void **) &d_strips[i], strips_cap * sizeof(TiffStrip)));
            CDS_CUDA(ctx, cudaEventCreateWithFlags(&up[i], cudaEventDisableTiming));
            CDS_CUDA(ctx, cudaEventCreateWithFlags(&decoded[i], cudaEventDisableTiming));
        }
        std::vector<TiffStrip> strips;
        int64_t calls = 0;
        return maskset_append(ms, n, mask_size_out, [&](int i0, int cnt, uint8_t *stage, cudaStream_t stream) -> cds_status {
            const int slot = (int) (calls & 1);
            CDS_TRY(collect_chunk(ctx, "cds_maskset_add_tiff", blob, offsets, i0, cnt, W, H, strips));
            const size_t bytes = (size_t) (offsets[i0 + cnt] - offsets[i0]);
            if (bytes > comp_cap || strips.size() > strips_cap) return ctx->fail(CDS_ERR_CAPACITY, "cds_maskset_add_tiff: internal staging too small");
            if (calls >= 2) CDS_CUDA(ctx, cudaStreamWaitEvent(h2d, decoded[slot], 0));       // the slot's previous files have been decoded
            CDS_CUDA(ctx, cudaMemcpyAsync(d_comp[slot], blob + offsets[i0], bytes, cudaMemcpyHostToDevice, h2d));
            // (the table is pageable host memory: the runtime stages it before the call returns, so `strips` may be reused)
            CDS_CUDA(ctx, cudaMemcpyAsync(d_strips[slot], strips.data(), strips.size() * sizeof(TiffStrip), cudaMemcpyHostToDevice, h2d));
            CDS_CUDA(ctx, cudaEventRecord(up[slot], h2d));
            ctx->stats.h2d_bytes += (int64_t) bytes + (int64_t) (strips.size() * sizeof(TiffStrip));
            CDS_CUDA(ctx, cudaStreamWaitEvent(stream, up[slot], 0));
            launch_tiff_decode(d_comp[slot], d_strips[slot], (int64_t) strips.size(), stage, stream);
            ctx->stats.kernel_launches++;
            CDS_CUDA(ctx, cudaGetLastError());
            CDS_CUDA(ctx, cudaEventRecord(decoded[slot], stream));
            calls++;
            return CDS_OK;
        });
    });
}


// Test hook: n TIFF files -> the code planes (and per-sector valid bits) a streaming search would build from them, through either
// ingest path, so that the fused kernel can be compared word for word with decode + encode and with the encoder's colour table.
extern "C" cds_status cds_debug_tiff_codes(cds_ctx *ctx, const uint8_t *blob, const int64_t *offsets, int64_t n, int32_t width, int32_t height,
                                           int32_t data_threshold, int32_t fused, uint32_t *codes_out, uint32_t *valid_out)
{
    return cds::abi_guard("cds_debug_tiff_codes", [&]() -> cds_status {
        if (!ctx) { set_tls_error("cds_debug_tiff_codes: NULL context"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (n < 0 || width <= 0 || height <= 0 || width > 2048 || height > 16384) return ctx->fail(CDS_ERR_BAD_ARG, "cds_debug_tiff_codes: bad size");
        if (n == 0) return CDS_OK;
        if (!blob || !offsets || !codes_out) return ctx->fail(CDS_ERR_BAD_ARG, "cds_debug_tiff_codes: NULL argument");
        DevState &ds = ctx->devs[0];
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        PlaneGeom g;
        g.W = width; g.H = height; g.pitch = choose_pitch(width); g.guard = CDS_GUARD_ROWS;
        const int vp = occupancy_valid_pitch(width);
        const size_t img_bytes = (size_t) width * height * 3;
        const size_t valid_words = (size_t) height * CDS_NUM_SECTORS * vp;
        uint8_t *d_comp = nullptr, *d_rgb = nullptr;
        TiffStrip *d_strips = nullptr;
        uint32_t *d_planes = nullptr, *d_valid = nullptr;
        unsigned long long *d_counter = nullptr;
        auto release = [&]() { cudaStreamSynchronize(ds.stream); for (void *p : {(void *) d_comp, (void *) d_rgb, (void *) d_strips, (void *) d_planes, (void *) d_valid, (void *) d_counter}) ds.pool.free(p); };
        struct Guard { std::function<void()> f; ~Guard() { f(); } } guard{release};
        std::vector<TiffStrip> strips;
        std::string err;
        for (int64_t i = 0; i < n; i++) {
            const int64_t a = offsets[i], b = offsets[i + 1];
            if (a < 0 || b < a) return ctx->fail(CDS_ERR_BAD_ARG, "cds_debug_tiff_codes: offsets must be non-decreasing");
            cds_status st = tiff_collect_strips(blob + a, (size_t) (b - a), width, height, (uint64_t) (a - offsets[0]),
                                                fused ? (uint64_t) i * height : (uint64_t) i * img_bytes, strips, err, fused != 0);
            if (st != CDS_OK) return ctx->fail(st, "cds_debug_tiff_codes: file " + std::to_string(i) + ": " + err);
        }
        const size_t comp_bytes = (size_t) (offsets[n] - offsets[0]);
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_comp, comp_bytes + 64));
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_strips, strips.size() * sizeof(TiffStrip) + 16));
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_planes, g.total_words(n) * sizeof(uint32_t)));
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_valid, (size_t) n * valid_words * sizeof(uint32_t)));
        if (!fused) CDS_CUDA(ctx, ds.pool.alloc((void **) &d_rgb, (size_t) n * img_bytes + 64));
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_counter, 64));
        CDS_CUDA(ctx, cudaMemcpyAsync(d_comp, blob + offsets[0], comp_bytes, cudaMemcpyHostToDevice, ds.stream));
        CDS_CUDA(ctx, cudaMemcpyAsync(d_strips, strips.data(), strips.size() * sizeof(TiffStrip), cudaMemcpyHostToDevice, ds.stream));
        launch_fill_words(d_planes, g.total_words(n), CDS_CODE_PAD_WORD, ds.stream);
        if (fused) {
            launch_tiff_encode(d_comp, d_strips, (int64_t) strips.size(), d_planes, g, 0, ds.d_rank_tab, data_threshold, d_valid, d_counter, ds.stream);
        } else {
            CDS_CUDA(ctx, cudaMemsetAsync(d_rgb, 0, (size_t) n * img_bytes, ds.stream));
            launch_tiff_decode(d_comp, d_strips, (int64_t) strips.size(), d_rgb, ds.stream);
            launch_encode_rgb(d_rgb, n, d_planes, g, 0, ds.d_rank_tab, data_threshold, ds.stream, d_valid);
        }
        CDS_CUDA(ctx, cudaGetLastError());
        for (int64_t i = 0; i < n; i++)
            CDS_CUDA(ctx, cudaMemcpy2DAsync(codes_out + (size_t) i * width * height, (size_t) width * 4, d_planes + g.row_offset(i, 0), (size_t) g.pitch * 4,
                                           (size_t) width * 4, (size_t) height, cudaMemcpyDeviceToHost, ds.stream));
        if (valid_out) CDS_CUDA(ctx, cudaMemcpyAsync(valid_out, d_valid, (size_t) n * valid_words * sizeof(uint32_t), cudaMemcpyDeviceToHost, ds.stream));
        CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
        return CDS_OK;
    });
}

// Test hook: per-sector valid bits [n][height][sectors][occupancy_valid_pitch(width)] -> the occupancy tile rows a search builds from
// them, [n][tile rows][occupancy_row_pitch] (sector rows, OR row, non-empty bits), so that the occupancy kernels can be compared
// with each other (cds_ctx_set_option "occupancy_kernel") and with the definition.
extern "C" cds_status cds_debug_occupancy(cds_ctx *ctx, const uint32_t *valid, int64_t n, int32_t width, int32_t height, int32_t xy_shift,
                                          uint32_t *occ_out)
{
    return cds::abi_guard("cds_debug_occupancy", [&]() -> cds_status {
        if (!ctx) { set_tls_error("cds_debug_occupancy: NULL context"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (n < 0 || width <= 0 || height <= 0 || width > 16384 || height > 16384 || xy_shift < 0 || xy_shift > 4 || (xy_shift & 1))
            return ctx->fail(CDS_ERR_BAD_ARG, "cds_debug_occupancy: bad size or xy_shift");
        if (n == 0) return CDS_OK;
        if (!valid || !occ_out) return ctx->fail(CDS_ERR_BAD_ARG, "cds_debug_occupancy: NULL argument");
        DevState &ds = ctx->devs[0];
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        PlaneGeom g;
        g.W = width; g.H = height; g.pitch = choose_pitch(width); g.guard = CDS_GUARD_ROWS;
        const int vp = occupancy_valid_pitch(width), tp = occupancy_tile_pitch(width);
        const size_t valid_words = (size_t) n * height * CDS_NUM_SECTORS * vp;
        const size_t occ_words = (size_t) n * occupancy_target_words(width, height);
        uint32_t *d_valid = nullptr, *d_occ = nullptr;
        auto release = [&]() { cudaStreamSynchronize(ds.stream); ds.pool.free(d_valid); ds.pool.free(d_occ); };
        struct Guard { std::function<void()> f; ~Guard() { f(); } } guard{release};
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_valid, valid_words * sizeof(uint32_t)));
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_occ, occ_words * sizeof(uint32_t)));
        CDS_CUDA(ctx, cudaMemcpyAsync(d_valid, valid, valid_words * sizeof(uint32_t), cudaMemcpyHostToDevice, ds.stream));
        CDS_CUDA(ctx, cudaMemsetAsync(d_occ, 0xA5, occ_words * sizeof(uint32_t), ds.stream));      // every word must be written by the kernels
        launch_occupancy(nullptr, g, 0, n, xy_shift / 2, tp, d_valid, n, d_occ, ds.stream, true);
        CDS_CUDA(ctx, cudaGetLastError());
        // the hook's layout (cdsgpu.h): sector rows, OR row, non-empty bits -- the rank-band bytes need code planes and are left out
        const int rowpitch = occupancy_row_pitch(tp), nzw = occupancy_nz_words(tp), out_pitch = (CDS_NUM_SECTORS + 1) * tp + nzw;
        const size_t rows = (size_t) n * occupancy_tile_rows(height);
        auto part = [&](int dst_col, int src_col, int words) {
            return cudaMemcpy2DAsync(occ_out + dst_col, (size_t) out_pitch * 4, d_occ + src_col, (size_t) rowpitch * 4, (size_t) words * 4, rows,
                                     cudaMemcpyDeviceToHost, ds.stream);
        };
        CDS_CUDA(ctx, part(0, 0, CDS_NUM_SECTORS * tp));
        CDS_CUDA(ctx, part(CDS_NUM_SECTORS * tp, occupancy_any_offset(tp), tp));
        CDS_CUDA(ctx, part((CDS_NUM_SECTORS + 1) * tp, occupancy_nz_offset(tp), nzw));
        CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
        return CDS_OK;
    });
}

// ------------------------------------------------------------------------------------------------------------------ PNG scanlines
// The device side of the PNG ingest: the host has inflated the zlib stream (cds_formats.cpp); what is left per image is
// height scanlines of [filter type][width * bps bytes], each filtered against the reconstructed bytes to the left and above
// (PNG specification, section 9: None, Sub, Up, Average, Paeth), samples big-endian.  One warp per image walks the rows in order
// with the previous reconstructed row in shared memory: None and Up are plain parallel passes, Sub is a prefix sum per byte lane
// (segments per lane + a warp scan), Average and Paeth are serial in x but independent per byte lane, so bps lanes run them.
// The reference's gradient files use filter None on every row (ImageJ's writer); the others are here for completeness.
namespace {

constexpr int kPngWarps = 4;

__global__ void __launch_bounds__(kPngWarps * 32)
png_unfilter_kernel(const uint8_t *__restrict__ filtered, size_t stride, const uint8_t *__restrict__ bytes_per_sample, int64_t n, int W, int H,
                    uint16_t *__restrict__ out, int row_buf)
{
    extern __shared__ uint8_t s_png[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t img = (int64_t) blockIdx.x * kPngWarps + warp;
    if (img >= n) return;
    uint8_t *cur = s_png + (size_t) warp * 2 * row_buf, *prev = cur + row_buf;
    const int bps = bytes_per_sample[img];
    const int rb = W * bps;
    const uint8_t *src = filtered + (size_t) img * stride;
    uint16_t *dst = out + (size_t) img * W * H;
    for (int i = lane; i < rb; i += 32) prev[i] = 0;
    __syncwarp();
    for (int y = 0; y < H; y++) {
        const uint8_t *line = src + (size_t) y * (1 + rb);
        const int f = line[0];
        const uint8_t *x = line + 1;
        if (f == 0) {
            for (int i = lane; i < rb; i += 32) cur[i] = x[i];
        } else if (f == 2) {
            for (int i = lane; i < rb; i += 32) cur[i] = (uint8_t) (x[i] + prev[i]);
        } else if (f == 1) {
            // Sub: recon[i] = x[i] + recon[i - bps]: a running sum per byte lane.  Lane l owns pixels [l * seg, (l + 1) * seg).
            const int seg = (W + 31) / 32;
            const int p0 = min(lane * seg, W), p1 = min(p0 + seg, W);
            uint32_t tot[2] = {0u, 0u};
            for (int px = p0; px < p1; px++)
                for (int b = 0; b < bps; b++) { tot[b] = (tot[b] + x[px * bps + b]) & 0xFFu; cur[px * bps + b] = (uint8_t) tot[b]; }
            uint32_t off[2];
            for (int b = 0; b < 2; b++) {
                uint32_t incl = tot[b];
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t u = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += u;
                }
                off[b] = (incl - tot[b]) & 0xFFu;
            }
            for (int px = p0; px < p1; px++)
                for (int b = 0; b < bps; b++) cur[px * bps + b] = (uint8_t) (cur[px * bps + b] + off[b]);
        } else if (f == 3 || f == 4) {
            if (lane < bps) {
                int a = 0, c = 0;                                   // reconstructed byte to the left, and above-left
                for (int i = lane; i < rb; i += bps) {
                    const int b = prev[i];
                    int pred;
                    if (f == 3) pred = (a + b) >> 1;
                    else { const int p = a + b - c, pa = abs(p - a), pb = abs(p - b), pc = abs(p - c); pred = (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c); }
                    a = (x[i] + pred) & 0xFF;
                    cur[i] = (uint8_t) a;
                    c = b;
                }
            }
        } else {
            for (int i = lane; i < rb; i += 32) cur[i] = 0;         // not a PNG filter type: the row stays black
        }
        __syncwarp();
        uint16_t *orow = dst + (size_t) y * W;
        if (bps == 2) for (int px = lane; px < W; px += 32) orow[px] = (uint16_t) ((uint32_t) cur[2 * px] << 8 | cur[2 * px + 1]);
        else for (int px = lane; px < W; px += 32) orow[px] = cur[px];
        uint8_t *t = cur; cur = prev; prev = t;
        __syncwarp();
    }
}

}  // namespace

void cds::launch_png_unfilter(const uint8_t *filtered, size_t stride, const uint8_t *bytes_per_sample, int64_t n, int width, int height,
                              uint16_t *out, cudaStream_t s)
{
    if (n <= 0) return;
    const int row_buf = (width * 2 + 15) / 16 * 16;
    const size_t smem = (size_t) kPngWarps * 2 * row_buf;
    png_unfilter_kernel<<<(unsigned) ((n + kPngWarps - 1) / kPngWarps), kPngWarps * 32, smem, s>>>(filtered, stride, bytes_per_sample, n, width, height, out, row_buf);
}

namespace cds {
// Inflates PNG files [first, first + cnt) of the blob into `h_filtered` (image i at i * stride, pinned or not) on up to `threads` host
// threads; bps[i] = bytes per sample.  The first failure is reported with its file number.
cds_status png_inflate_many(cds_ctx *ctx, const char *who, const uint8_t *blob, const int64_t *offsets, const int64_t *which, int64_t cnt,
                            int W, int H, uint8_t *h_filtered, size_t stride, uint8_t *bps)
{
    const int threads = (int) std::max<int64_t>(1, std::min<int64_t>(cnt, std::min<unsigned>(32u, std::max(1u, std::thread::hardware_concurrency()))));
    std::vector<cds_status> st(threads, CDS_OK);
    std::vector<std::string> errs(threads);
    std::vector<int64_t> bad(threads, -1);
    auto body = [&](int t) {
        for (int64_t i = t; i < cnt; i += threads) {
            const int64_t f = which ? which[i] : i;
            const int64_t a = offsets[f], b = offsets[f + 1];
            int depth = 16;
            std::string err;
            cds_status s = (a < 0 || b < a) ? CDS_ERR_BAD_ARG : png_inflate(blob + a, (size_t) (b - a), W, H, &depth, h_filtered + (size_t) i * stride, stride, err);
            if (s != CDS_OK) { if (st[t] == CDS_OK) { st[t] = s; errs[t] = err.empty() ? "offsets must be non-decreasing" : err; bad[t] = f; } continue; }
            bps[i] = (uint8_t) (depth / 8);
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; t++) pool.emplace_back(body, t);
    body(0);
    for (auto &th : pool) th.join();
    for (int t = 0; t < threads; t++)
        if (st[t] != CDS_OK) return ctx->fail(st[t], std::string(who) + ": file " + std::to_string(bad[t]) + ": " + errs[t]);
    return CDS_OK;
}
}  // namespace cds

extern "C" cds_status cds_png_decode_gray16(cds_ctx *ctx, const uint8_t *blob, const int64_t *offsets, int64_t n, int32_t width, int32_t height, uint16_t *out)
{
    return cds::abi_guard("cds_png_decode_gray16", [&]() -> cds_status {
        if (!ctx) { set_tls_error("cds_png_decode_gray16: NULL context"); return CDS_ERR_BAD_ARG; }
        std::lock_guard<std::recursive_mutex> lk(ctx->mu);
        if (n < 0 || width <= 0 || height <= 0 || width > 16384 || height > 16384) return ctx->fail(CDS_ERR_BAD_ARG, "cds_png_decode_gray16: bad size");
        if (n == 0) return CDS_OK;
        if (!blob || !offsets || !out) return ctx->fail(CDS_ERR_BAD_ARG, "cds_png_decode_gray16: NULL argument");
        ctx->stats = cds_search_stats{};
        DevState &ds = ctx->devs[0];
        CDS_CUDA(ctx, cudaSetDevice(ds.dev));
        const size_t stride = ((size_t) height * (1 + (size_t) width * 2) + 15) / 16 * 16;
        const size_t px = (size_t) width * height;
        const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(64, (int64_t) (((size_t) 256 << 20) / stride)));
        CDS_TRY(ctx->ensure_pinned(ds, (size_t) chunk * (stride + 16)));
        uint8_t *h_f = (uint8_t *) ds.h_pinned, *h_bps = h_f + (size_t) chunk * stride;
        uint8_t *d_f = nullptr, *d_bps = nullptr;
        uint16_t *d_out = nullptr;
        auto release = [&]() { cudaStreamSynchronize(ds.stream); ds.pool.free(d_f); ds.pool.free(d_bps); ds.pool.free(d_out); };
        struct Guard { std::function<void()> f; ~Guard() { f(); } } guard{release};
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_f, (size_t) chunk * stride));
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_bps, (size_t) chunk));
        CDS_CUDA(ctx, ds.pool.alloc((void **) &d_out, (size_t) chunk * px * sizeof(uint16_t)));
        // device inflate (cds_inflate.cu): the files' zlib streams are uploaded as stored; the pinned staging area (sized for scanlines)
        // holds {jobs, bytes per sample, streams, statuses} with room to spare
        uint8_t *d_z = nullptr;
        int32_t *d_stat = nullptr;
        const size_t z_head = ((size_t) chunk * (sizeof(InflateJob) + 1) + 15) / 16 * 16, z_stat = (size_t) chunk * sizeof(int32_t);
        const size_t z_cap = (size_t) chunk * (stride + 16) - z_head - z_stat;
        auto release_z = [&]() { cudaStreamSynchronize(ds.stream); ds.pool.free(d_z); ds.pool.free(d_stat); };
        Guard guard_z{release_z};
        if (ctx->device_inflate) {
            CDS_CUDA(ctx, ds.pool.alloc((void **) &d_z, z_head + z_cap));
            CDS_CUDA(ctx, ds.pool.alloc((void **) &d_stat, z_stat));
        }
        for (int64_t i0 = 0; i0 < n; i0 += chunk) {
            const int64_t cnt = std::min(chunk, n - i0);
            bool inflated = false;
            if (ctx->device_inflate) {
                InflateJob *h_jobs = (InflateJob *) h_f;
                uint8_t *h_b = h_f + (size_t) chunk * sizeof(InflateJob), *h_z = h_f + z_head;
                int32_t *h_stat = (int32_t *) (h_f + z_head + z_cap);
                size_t zo = 2;                                     // deflate data (behind the 2-byte zlib header) on 4-byte boundaries
                bool staged = true;
                for (int64_t i = 0; i < cnt && staged; i++) {
                    const int64_t a = offsets[i0 + i], b = offsets[i0 + i + 1];
                    std::string err;
                    size_t used = 0;
                    if (a < 0 || b < a) return ctx->fail(CDS_ERR_BAD_ARG, "cds_png_decode_gray16: offsets must be non-decreasing");
                    const cds_status ps = png_collect_idat(blob + a, (size_t) (b - a), width, height, h_z + zo, z_cap - zo, z_head + zo, &used, &h_jobs[i], &h_b[i], err);
                    if (ps == CDS_ERR_CAPACITY) { staged = false; break; }      // streams larger than their images: the host path takes the chunk
                    if (ps != CDS_OK) return ctx->fail(ps, "cds_png_decode_gray16: file " + std::to_string(i0 + i) + ": " + err);
                    zo = (zo + used + 1) / 4 * 4 + 2;
                    if (zo > z_cap) { staged = false; break; }
                }
                if (staged) {
                    CDS_CUDA(ctx, cudaMemcpyAsync(d_z, h_f, z_head + zo, cudaMemcpyHostToDevice, ds.stream));
                    const uint8_t *d_b = d_z + (size_t) chunk * sizeof(InflateJob);
                    launch_png_inflate(d_z, (const InflateJob *) d_z, cnt, d_f, stride, d_b, width, height, d_stat, ds.stream);
                    CDS_CUDA(ctx, cudaMemcpyAsync(h_stat, d_stat, (size_t) cnt * sizeof(int32_t), cudaMemcpyDeviceToHost, ds.stream));
                    CDS_CUDA(ctx, cudaMemcpyAsync(d_bps, d_b, (size_t) cnt, cudaMemcpyDeviceToDevice, ds.stream));
                    CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
                    ctx->stats.kernel_launches++;
                    // refused streams: zlib on the host decides, and its scanlines replace the device's
                    std::vector<uint8_t> lines;
                    for (int64_t i = 0; i < cnt; i++) {
                        if (h_stat[i] == 0 && !(ctx->device_inflate == 2 && (i & 1))) continue;
                        lines.resize(stride);
                        std::string err;
                        int depth = 16;
                        const cds_status ps = png_inflate(blob + offsets[i0 + i], (size_t) (offsets[i0 + i + 1] - offsets[i0 + i]), width, height, &depth, lines.data(), stride, err);
                        if (ps != CDS_OK) return ctx->fail(ps, "cds_png_decode_gray16: file " + std::to_string(i0 + i) + ": " + err);
                        CDS_CUDA(ctx, cudaMemcpy(d_f + (size_t) i * stride, lines.data(), stride, cudaMemcpyHostToDevice));
                        ctx->stats.host_inflate_fallbacks++;
                    }
                    inflated = true;
                }
            }
            if (!inflated) {
                CDS_TRY(png_inflate_many(ctx, "cds_png_decode_gray16", blob, offsets + i0, nullptr, cnt, width, height, h_f, stride, h_bps));
                CDS_CUDA(ctx, cudaMemcpyAsync(d_f, h_f, (size_t) cnt * stride, cudaMemcpyHostToDevice, ds.stream));
                CDS_CUDA(ctx, cudaMemcpyAsync(d_bps, h_bps, (size_t) cnt, cudaMemcpyHostToDevice, ds.stream));
            }
            launch_png_unfilter(d_f, stride, d_bps, cnt, width, height, d_out, ds.stream);
            CDS_CUDA(ctx, cudaGetLastError());
            CDS_CUDA(ctx, cudaMemcpyAsync(out + (size_t) i0 * px, d_out, (size_t) cnt * px * sizeof(uint16_t), cudaMemcpyDeviceToHost, ds.stream));
            CDS_CUDA(ctx, cudaStreamSynchronize(ds.stream));
            ctx->stats.kernel_launches++;
        }
        return CDS_OK;
    });
}

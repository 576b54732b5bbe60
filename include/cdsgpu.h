/*
 * cdsgpu.h -- C ABI of the B200-native colour-depth MIP matching library (libcdsgpu.so).
 *
 * This is the drop-in boundary for ONE hot path of JaneliaSciComp/colormipsearch v3.1.1:
 *   - pixel-match colour depth search  (PixelMatchColorDepthSearchAlgorithm)
 *   - 2D shape / gradient-area-gap score (Shape2DMatchColorDepthSearchAlgorithm)
 * The reference is pure Java and has no FFI of its own; these entry points are what a JNI or
 * Panama-FFM binding behind its ColorDepthSearchAlgorithmProvider / ColorDepthSearchAlgorithm /
 * ColorMIPSearchProcessor interfaces calls (INTEGRATION.md shows the binding).  Every function
 * cites the reference interface it replaces; API/ abbreviates
 * colormipsearch-api/src/main/java/org/janelia/colormipsearch/ and TOOLS/ abbreviates
 * colormipsearch-tools/src/main/java/org/janelia/colormipsearch/cmd/.
 *
 * Conventions
 *   - plain C types only; every pointer is caller-owned HOST memory; calls block until results are
 *     in the caller's buffers; nothing retains caller pointers after return.
 *   - every function returns a cds_status; on failure cds_last_error() has the message.  Nothing
 *     aborts or throws across the ABI.  CDS_ERR_BAD_ARG / CDS_ERR_SIZE_MISMATCH correspond to the
 *     reference's IllegalArgumentException sites, everything else to IllegalStateException.
 *   - there is NO CPU fallback: without a CUDA device cds_ctx_create fails with CDS_ERR_NO_DEVICE.
 *   - images: RGB = uint8[H][W][3] in R,G,B order (API/imageprocessing/ColorImageArray.java:6-31),
 *     gray16 = uint16[H][W] (ShortImageArray.java:4-16), gray8 = uint8[H][W] (ByteImageArray.java:3-16).
 *   - a cds_ctx may be used from several host threads; calls on one ctx are serialised internally (cds_pairq_score is the exception:
 *     it takes no context-wide lock).  Searches, library / mask-set construction, the shape score and the pair queue use every device
 *     of the context; the one-shot utilities (cds_make_zgap, cds_tiff_decode_rgb, cds_png_decode_gray16, the cds_debug_* hooks) run on
 *     its first device.
 */
#ifndef CDSGPU_H
#define CDSGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden; these are its only exports */
#endif

#define CDSGPU_ABI_VERSION 2   /* 2: cds_search_stats grew by host_inflate_fallbacks (callers pass their own struct: sizes must agree) */

typedef int32_t cds_status;
enum {
    CDS_OK = 0,
    CDS_ERR_BAD_ARG = 1,        /* IllegalArgumentException: odd xyShift (API/cds/ColorDepthSearchAlgorithmProviderFactory.java:57-60), bad sizes, null pointers */
    CDS_ERR_SIZE_MISMATCH = 2,  /* IllegalArgumentException: image size differs from the query's (API/cds/PixelMatchColorDepthSearchAlgorithm.java:171-175) */
    CDS_ERR_NO_DEVICE = 3,      /* no CUDA device / device id out of range */
    CDS_ERR_CUDA = 4,           /* a CUDA runtime call or kernel failed */
    CDS_ERR_OOM = 5,            /* device or host allocation failed */
    CDS_ERR_CAPACITY = 6,       /* library / mask set is full */
    CDS_ERR_UNSUPPORTED = 7     /* parameter combination outside the supported envelope (documented per call) */
};

typedef struct cds_ctx cds_ctx;
typedef struct cds_library cds_library;
typedef struct cds_maskset cds_maskset;
typedef struct cds_shape_maskset cds_shape_maskset;

/* Half-open rectangle [x0,x1) x [y0,y1): one label region excluded from matching
 * (TOOLS/AbstractColorDepthMatchArgs.java:101-119 getRegionGeneratorForTextLabels;
 *  API/imageprocessing/ImageRegionDefinition.java). */
typedef struct cds_rect { int32_t x0, y0, x1, y1; } cds_rect;

#define CDS_MAX_RECTS 8

/* Parameters of the pixel-match provider: the arguments of
 * ColorDepthSearchAlgorithmProviderFactory.createPixMatchCDSAlgorithmProvider
 * (API/cds/ColorDepthSearchAlgorithmProviderFactory.java:30-74) plus the query threshold that
 * createColorDepthSearchAlgorithm receives per mask (:45-48). */
typedef struct cds_pixparams {
    int32_t mask_threshold;     /* queryThreshold: mask pixel kept when R|G|B > threshold (API/cds/AbstractColorDepthSearchAlgorithm.java:116) */
    int32_t data_threshold;     /* targetThreshold / dataThreshold (API/cds/PixelMatchColorDepthSearchAlgorithm.java:250) */
    double  z_tolerance;        /* pixColorFluctuation / 100 (ProviderFactory :55-56); must be < 1000 */
    int32_t xy_shift;           /* even, 0..CDS_MAX_XY_SHIFT; 0 and 2 are the values the Java reference can run (see oracle) */
    int32_t mirror;             /* mirrorMask */
    int32_t n_rects;            /* 0..CDS_MAX_RECTS */
    cds_rect rects[CDS_MAX_RECTS];
} cds_pixparams;

#define CDS_MAX_XY_SHIFT 8

/* ---------------------------------------------------------------- context ---------------------------------------------------------------- */

/* Create a context over n_dev CUDA devices (device_ids may be NULL = devices 0..n_dev-1; n_dev = 0 = all visible).
 * Replaces: nothing in the reference (it has no device); lifetime = one ColorDepthSearchAlgorithmProvider / one command run. */
cds_status cds_ctx_create(const int32_t *device_ids, int32_t n_dev, cds_ctx **out);
void       cds_ctx_destroy(cds_ctx *ctx);
int32_t    cds_ctx_num_devices(const cds_ctx *ctx);
/* Message of the last failing call on this thread (ctx may be NULL for cds_ctx_create failures). Never NULL. */
const char *cds_last_error(const cds_ctx *ctx);
int32_t    cds_abi_version(void);
/* Tuning / test switches.  "match_kernel": 0 = automatic (default), 1 = candidate kernel, 2 = band kernel, 3 = gather kernel;
 * a kernel that does not support the search's parameters falls through to the next one.  All three compute the same
 * scores bit for bit (tests/test_pixelmatch_gpu.py cross-checks them).
 * "stream_chunk": targets per chunk of the chunked searches (default 256).
 * "stream_chunk_tiff": most targets per chunk of cds_search_stream_tiff (default 4096: the match kernel hands out whole targets to its
 *   persistent CTAs, so long chunks keep its grid full; the first chunks of a call are 256, 512, ... files so that matching starts early).
 * "resident_occupancy": 1 (default) keeps a library's occupancy bitmaps on the device next to its code planes (+23 % memory) and
 * falls back to building them per target chunk inside cds_search_topk when they do not fit; 0 always builds them per chunk.
 * "stream_chunk_bytes": most file bytes per chunk of cds_search_stream_tiff (default and maximum 3 GiB; a chunk also ends there).
 * "fused_ingest": 1 (default) = the streaming searches over TIFF files turn the strips straight into the library's code words;
 * 0 = decode to RGB pixels first, then encode (the two-kernel path, kept as a cross-check).
 * "cand_wait_mode", "cand_l2_hint", "cand_warps", "cand_stages", "cand_max_rows": tuning knobs of the candidate kernel (csrc/cds_cand.cuh),
 *   process-wide.  "occupancy_kernel": 1 (default) = the single-pass occupancy kernel for xyShift 2, 0 = the generic one (cross-check).
 * "device_inflate": 1 (default) = cds_shape_score_pairs_files uploads the gradient PNG files as stored and inflates their zlib streams
 *   on the device, one warp per stream (csrc/cds_inflate.h); 0 = host threads inflate them (zlib) and the scanlines are uploaded;
 *   2 (tests) = like 1, with every odd image of a window treated as refused.  cds_png_decode_gray16 follows the same switch.
 *   Same pixels either way: a stream the device refuses is read by zlib on the host (host_inflate_fallbacks in the stats).
 * "shape_inflate_window": most targets per window of cds_shape_score_pairs_files when the gradient streams are inflated on the device
 *   (0 = default 2048; halved until every device has two windows; a window's buffers are ~10 MB per target).
 * "wide_lists": 1 = mask sets prepared from now on carry each mask pixel's rank interval in the candidate kernel's lists (4 bytes per
 *   pixel and list) instead of a reference into a per-group palette (2 bytes).  0 (default): only sets with a group of more than
 *   2 047 colour classes do (brightness-scaled LM images as masks -- the reverse search); scores are the same either way.
 * "best_list_bytes": most bytes per device of the list of passing pairs that the *_best_matches searches keep on the device (12 bytes per
 *   pair; default 1 GiB, 12 .. 4 GiB).  While it runs, the selection over the list takes about 144 bytes more per pair on the first device
 *   (all devices' lists together) and a compaction about 96; a call that would not fit in the device's free memory returns CDS_ERR_OOM
 *   naming the bytes it needs.
 * Unknown names: CDS_ERR_BAD_ARG. */
cds_status cds_ctx_set_option(cds_ctx *ctx, const char *name, int64_t value);

/* Pinned host memory for callers that want full-rate uploads (optional; any host pointer is accepted everywhere). */
cds_status cds_host_alloc(cds_ctx *ctx, uint64_t bytes, void **out);
cds_status cds_host_free(cds_ctx *ctx, void *p);

/* ---------------------------------------------------------------- target library --------------------------------------------------------- */

/* A device-resident library of target MIPs of one size, sharded block-cyclically over the context's devices.
 * Replaces: the Guava cache of decoded target ImageArrays (TOOLS/CachedMIPsUtils.java:60-110) that
 * LocalColorMIPSearchProcessor re-reads for every mask (TOOLS/cdsprocess/LocalColorMIPSearchProcessor.java:93-105). */
cds_status cds_library_create(cds_ctx *ctx, int32_t width, int32_t height, int64_t capacity, cds_library **out);
void       cds_library_destroy(cds_library *lib);
/* Append n RGB images (uint8[n][H][W][3]); *first_index (may be NULL) receives the index of the first one. */
cds_status cds_library_add_rgb(cds_library *lib, const uint8_t *rgb, int64_t n, int64_t *first_index);
/* Append n deterministic synthetic LM-like targets generated on the device (bench / scale tests); indices continue
 * from the current size and image i is synth target number (first_synth_index + i) of `seed`. */
cds_status cds_library_generate_synthetic(cds_library *lib, uint64_t seed, int64_t first_synth_index, int64_t n, int64_t *first_index);
int64_t    cds_library_size(const cds_library *lib);
cds_status cds_library_clear(cds_library *lib);   /* forget all targets, keep the allocation */

/* ---------------------------------------------------------------- pixel match ------------------------------------------------------------ */

/* A set of prepared query masks sharing one parameter set; replicated on every device.
 * Replaces: one PixelMatchColorDepthSearchAlgorithm per mask, i.e.
 * ColorDepthSearchAlgorithmProvider.createColorDepthSearchAlgorithm (API/cds/ColorDepthSearchAlgorithmProvider.java:20-32)
 * and the constructor work at API/cds/PixelMatchColorDepthSearchAlgorithm.java:29-101
 * (getMaskPosArray, generateShiftedMasks, mirrorMask).
 * Errors: CDS_ERR_BAD_ARG for odd xy_shift (Java: IllegalArgumentException), CDS_ERR_UNSUPPORTED for xy_shift > CDS_MAX_XY_SHIFT
 * or z_tolerance >= 1000. */
cds_status cds_maskset_create(cds_ctx *ctx, int32_t width, int32_t height, const cds_pixparams *params, cds_maskset **out);
void       cds_maskset_destroy(cds_maskset *ms);
/* Add n masks (uint8[n][H][W][3]).  mask_size_out[n] (may be NULL) receives getQuerySize() of each
 * (API/cds/AbstractColorDepthSearchAlgorithm.java:71-73).  An empty mask is legal (scores 0, :169-170). */
cds_status cds_maskset_add_rgb(cds_maskset *ms, const uint8_t *rgb, int32_t n, int32_t *mask_size_out);
int32_t    cds_maskset_size(const cds_maskset *ms);
cds_status cds_maskset_get_mask_sizes(const cds_maskset *ms, int32_t *sizes_out /* [M] */);

/* calculateMatchingScore of every mask against every target (API/cds/PixelMatchColorDepthSearchAlgorithm.java:166-219):
 * scores[m*T + t] = matching pixels, mirrored[m*T + t] = bestScoreMirrored (may be NULL).  T = cds_library_size(lib).
 * Used by the single-pair provider and by parity tests.  CDS_ERR_SIZE_MISMATCH when the library's image size differs. */
cds_status cds_search_dense(cds_ctx *ctx, const cds_maskset *ms, cds_library *lib, int32_t *scores, uint8_t *mirrored);

/* Per mask, the K best targets that pass ColorMIPSearch.isMatch (API/cds/ColorMIPSearch.java:42-45:
 * score > 0 && (float)(score/maskSize) > pct_positive_pixels/100), ordered by score descending, ties by ascending target
 * index (= a single-threaded run of TOOLS/cdsprocess/LocalColorMIPSearchProcessor.java:55-116 followed by the
 * stable sort of TOOLS/ColorDepthSearchCmd.java:403-409).  Selection happens on the devices; per-device lists are merged on
 * the host.  out_score/out_target/out_mirrored are [M][K]; out_count[m] = entries filled for mask m (<= K). */
cds_status cds_search_topk(cds_ctx *ctx, const cds_maskset *ms, cds_library *lib, int32_t k, double pct_positive_pixels,
                           int32_t *out_score, int64_t *out_target, uint8_t *out_mirrored, int32_t *out_count);

/* The batched seam: ColorMIPSearchProcessor.findAllColorDepthMatches(masks, targets)
 * (TOOLS/cdsprocess/ColorMIPSearchProcessor.java:8-12, LocalColorMIPSearchProcessor.java:55-116) for targets held in HOST memory
 * that need not stay on the devices: targets_rgb is uint8[n_targets][H][W][3]; the result is what cds_library_add_rgb of all of
 * them followed by cds_search_topk would return (target = index into targets_rgb), but uploads, encoding and matching of
 * successive chunks overlap, and device memory use does not grow with n_targets.  Pinned memory (cds_host_alloc) gives full
 * PCIe rate; any host pointer works.  Image size = the mask set's. */
cds_status cds_search_stream_rgb(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *targets_rgb, int64_t n_targets,
                                 int32_t k, double pct_positive_pixels,
                                 int32_t *out_score, int64_t *out_target, uint8_t *out_mirrored, int32_t *out_count);

/* The same streaming search without a K: EVERY (mask, target) pair that passes ColorMIPSearch.isMatch -- what
 * LocalColorMIPSearchProcessor keeps (TOOLS/cdsprocess/LocalColorMIPSearchProcessor.java:93-105: filter(m -> m.isMatchFound())) --
 * ordered by mask, then descending matchingPixels, then ascending target (the stable sort of TOOLS/ColorDepthSearchCmd.java:403-409
 * after a single-threaded run).  out_* hold `capacity` entries; *out_count receives the number of passing pairs.  When more than
 * `capacity` pairs pass, nothing is written, *out_count still tells how many there are and the call returns CDS_ERR_CAPACITY. */
cds_status cds_search_stream_matches_rgb(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *targets_rgb, int64_t n_targets,
                                         double pct_positive_pixels, int64_t capacity,
                                         int32_t *out_mask, int64_t *out_target, int32_t *out_score, uint8_t *out_mirrored,
                                         int64_t *out_count);

/* Every pair that passes isMatch, for a device-resident library (same outputs and conventions as cds_search_stream_matches_rgb;
 * target = index in the library). */
cds_status cds_search_matches(cds_ctx *ctx, const cds_maskset *ms, cds_library *lib, double pct_positive_pixels, int64_t capacity,
                              int32_t *out_mask, int64_t *out_target, int32_t *out_score, uint8_t *out_mirrored, int64_t *out_count);

/* ---------------------------------------------------------------- image ingest (SURVEY 8f, row f4) ------------------------------------------- */

/* Colour-depth MIP libraries are stored as RGB TIFF files, normally PackBits-compressed (the reference's own fixtures: 1210x566,
 * 71 strips of 8 rows, 65-255 kB per 2 MB image).  The reference decodes them on the JVM: ImageJ's Opener for whole files
 * (API/imageprocessing/ImageArrayUtils.java:176-182) and its own strip loop + packBitsUncompress for PackBits files
 * (ImageArrayUtils.java:184-258, LocalTiffDecoder.java).  Here the container is parsed on the host (tags only), the strips
 * travel to the device AS STORED and are decoded there, so a search over host-resident files moves 8-30 x fewer bytes over PCIe.
 * Supported: classic (non-Big) TIFF, either byte order, first image of the file, 8-bit RGB chunky (SamplesPerPixel 3,
 * PlanarConfiguration 1), Compression 1 (none) or 32773 (PackBits), strips (no tiles).
 * Anything else: CDS_ERR_UNSUPPORTED naming the file (LZW, which the reference hands to ImageJ, included). */
typedef struct cds_tiff_info {
    int32_t width, height;
    int32_t compression;          /* tag 259: 1 none, 5 LZW, 32773 PackBits, ... */
    int32_t samples_per_pixel;    /* tag 277 */
    int32_t bits_per_sample;      /* tag 258 (first sample) */
    int32_t photometric;          /* tag 262 */
    int32_t planar_config;        /* tag 284 (1 when absent) */
    int32_t rows_per_strip;       /* tag 278 (height when absent) */
    int32_t n_strips;
    int32_t big_endian;           /* 1 for "MM" files */
    int64_t data_bytes;           /* sum of the strip byte counts */
    int32_t decodable;            /* 1 when the device decoder takes this file */
    int32_t pad;
} cds_tiff_info;

/* Host only (no device needed): reads the first IFD of a TIFF file held in memory. */
cds_status cds_tiff_probe(const uint8_t *file, int64_t len, cds_tiff_info *info);

/* Host only: writes an 8-bit RGB image as a little-endian TIFF with PackBits-compressed strips of rows_per_strip rows (every
 * row packed on its own, as the TIFF specification asks).  compression = 32773 or 1.  cds_tiff_encode_bound gives a capacity
 * that always suffices.  Used to build test and benchmark libraries; the reference only reads TIFFs. */
int64_t    cds_tiff_encode_bound(int32_t width, int32_t height, int32_t rows_per_strip);
cds_status cds_tiff_encode_rgb(const uint8_t *rgb, int32_t width, int32_t height, int32_t rows_per_strip, int32_t compression,
                               uint8_t *out, int64_t capacity, int64_t *out_len);

/* n TIFF files stored back to back in `blob`: file i is blob[offsets[i] .. offsets[i+1]) (offsets has n + 1 entries).
 * Decodes them on device 0 of the context and returns the pixels: out_rgb is uint8[n][height][width][3].  A strip that decodes
 * to fewer bytes than its rows need leaves the rest 0, like the zero-initialised array of ImageArrayUtils.java:198.
 * CDS_ERR_SIZE_MISMATCH when a file's size is not width x height. */
cds_status cds_tiff_decode_rgb(cds_ctx *ctx, const uint8_t *blob, const int64_t *offsets, int64_t n,
                               int32_t width, int32_t height, uint8_t *out_rgb);

/* cds_library_add_rgb / cds_maskset_add_rgb for TIFF files: compressed strips are uploaded and decoded on the devices. */
cds_status cds_maskset_add_tiff(cds_maskset *ms, const uint8_t *blob, const int64_t *offsets, int32_t n, int32_t *mask_size_out /* [n], may be NULL */);
cds_status cds_library_add_tiff(cds_library *lib, const uint8_t *blob, const int64_t *offsets, int64_t n, int64_t *first_index);

/* cds_search_stream_rgb / cds_search_stream_matches_rgb for targets that are TIFF files in host memory (same results as decoding
 * them first): per chunk the host parses the tags, the copy stream uploads the files' bytes as they are, and the compute stream
 * decodes, encodes and matches them.  Pinned memory (cds_host_alloc) for `blob` gives full PCIe rate. */
cds_status cds_search_stream_tiff(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *blob, const int64_t *offsets, int64_t n_targets,
                                  int32_t k, double pct_positive_pixels,
                                  int32_t *out_score, int64_t *out_target, uint8_t *out_mirrored, int32_t *out_count);
cds_status cds_search_stream_matches_tiff(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *blob, const int64_t *offsets, int64_t n_targets,
                                          double pct_positive_pixels, int64_t capacity,
                                          int32_t *out_mask, int64_t *out_target, int32_t *out_score, uint8_t *out_mirrored,
                                          int64_t *out_count);

/* ---- what the reference reads that is not a PackBits / stored RGB TIFF (csrc/cds_formats.cpp) ---- */

/* Host only.  Decodes the first image of any 8-bit RGB strip TIFF the tag parser understands -- uncompressed, PackBits, or LZW with or
 * without the horizontal predictor (tag 317) -- into out_rgb = uint8[height][width][3].  LZW files are what the reference hands to
 * ImageJ's Opener (API/imageprocessing/ImageArrayUtils.java:176-182, 196-198: every TIFF whose compression is not PackBits). */
cds_status cds_tiff_decode_rgb_host(const uint8_t *file, int64_t len, int32_t width, int32_t height, uint8_t *out_rgb);
/* Host only.  Rewrites such a file as the PackBits TIFF (strips of 8 rows) the device ingest takes, so that an LZW library can be fed
 * to cds_search_stream_tiff / cds_library_add_tiff after one pass on the host.  capacity >= cds_tiff_encode_bound(width, height, 8). */
cds_status cds_tiff_to_packbits(const uint8_t *file, int64_t len, uint8_t *out, int64_t capacity, int64_t *out_len);

/* PNG: the gradient images of gradientScores are 16-bit grayscale PNG files, which the reference reads through ImageIO.read
 * (API/imageprocessing/ImageArrayUtils.java:98-121, 176-178).  Supported: grayscale, 8 or 16 bits, not interlaced. */
typedef struct cds_png_info {
    int32_t width, height;
    int32_t bit_depth;            /* 8 or 16 for decodable files */
    int32_t color_type;           /* 0 = grayscale */
    int32_t interlace;
    int32_t decodable;
    int64_t data_bytes;           /* sum of the IDAT chunk lengths */
} cds_png_info;
cds_status cds_png_probe(const uint8_t *file, int64_t len, cds_png_info *info);      /* host only */
/* n PNG files stored back to back (blob / offsets as for the TIFF calls) -> out = uint16[n][height][width] (8-bit files are widened,
 * like ImageArray.get on a ByteImageArray).  The files are uploaded as stored; their zlib streams are inflated (one warp per stream,
 * csrc/cds_inflate.h), the scanline filters (None, Sub, Up, Average, Paeth) undone and the samples byte-swapped on device 0.  The image
 * is the first height * (1 + width * bytes per sample) bytes of the stream (data behind them is ignored, a shorter stream is an error;
 * the Adler-32 trailer is not checked).  A stream the device refuses is read by zlib on the host, which then has the last word
 * (cds_search_stats.host_inflate_fallbacks); "device_inflate" 0 (cds_ctx_set_option) inflates everything on host threads. */
cds_status cds_png_decode_gray16(cds_ctx *ctx, const uint8_t *blob, const int64_t *offsets, int64_t n, int32_t width, int32_t height, uint16_t *out);
/* Host only, test hook: raw DEFLATE data (RFC 1951, no zlib header) through the decoder that the device runs one warp per stream
 * (csrc/cds_inflate.h), built for a single lane.  *out_len = bytes produced; *reason (may be NULL) = 0 or why the stream was refused
 * (1 input ends early, 2 bad block, 3 bad code lengths, 4 bad symbol, 5 distance before the start, 6 more than `capacity` bytes). */
cds_status cds_debug_inflate_host(const uint8_t *in, int64_t len, uint8_t *out, int64_t capacity, int64_t *out_len, int32_t *reason);
/* Host only: a 16-bit grayscale PNG writer for tests and the bench (filter_mode 0..4 = that filter on every row, -1 = per row the
 * filter with the smallest sum of absolute differences).  cds_png_encode_bound gives a capacity that suffices. */
int64_t    cds_png_encode_bound(int32_t width, int32_t height);
cds_status cds_png_encode_gray16(const uint16_t *pixels, int32_t width, int32_t height, int32_t filter_mode,
                                 uint8_t *out, int64_t capacity, int64_t *out_len);

/* zip archives: libraries are routinely zip files whose entries are the MIPs (API/mips/NeuronMIPUtils.java:124-129, 177-227).
 * cds_zip_index reads the central directory (entries may be NULL with capacity 0 to count); a stored entry (method 0) IS the file:
 * archive + data_offset, `size` bytes -- a (blob, offsets) pair for the TIFF calls can point straight into the mapped archive when
 * the wanted entries are stored and consecutive; cds_zip_read copies (stored) or inflates (deflate) an entry and checks its CRC.
 * cds_zip_find looks an entry up like the reference: the exact name, else the first non-directory entry with the same file name
 * (NeuronMIPUtils.openZipEntryStream :193-208); -1 when there is none.  zip64 is not supported. */
typedef struct cds_zip_entry {
    int64_t name_offset;          /* the entry's name inside the archive (not NUL-terminated) */
    int32_t name_len;
    int32_t method;               /* 0 stored, 8 deflate */
    int64_t data_offset;
    int64_t compressed_size, size;
    uint32_t crc32;
    int32_t is_directory;
} cds_zip_entry;
cds_status cds_zip_index(const uint8_t *archive, int64_t len, cds_zip_entry *entries, int64_t capacity, int64_t *n_entries);
int64_t    cds_zip_find(const uint8_t *archive, const cds_zip_entry *entries, int64_t n_entries, const char *name);
cds_status cds_zip_read(const uint8_t *archive, int64_t len, const cds_zip_entry *entry, uint8_t *out, int64_t capacity);

/* One mask x one target held in host memory: the literal single-pair call of the Java API
 * (ColorDepthSearchAlgorithm.calculateMatchingScore, API/cds/ColorDepthSearchAlgorithm.java:60-61). */
cds_status cds_score_pair_rgb(cds_ctx *ctx, const cds_maskset *ms, int32_t mask_index, const uint8_t *target_rgb,
                              int32_t target_width, int32_t target_height,
                              int32_t *score_out, double *ratio_out, int32_t *mirrored_out);

/* The single-pair call at scale: a micro-batching scorer with a device-side target cache.
 * The reference makes one calculateMatchingScore call per (mask, target) pair from ~40 pool threads at once, on one algorithm
 * instance per mask (TOOLS/cdsprocess/LocalColorMIPSearchProcessor.java:93-105), and the SAME target image recurs across masks
 * because targets come out of a cache (TOOLS/CachedMIPsUtils.java:60-110).  cds_pairq_score is that call: it blocks its caller
 * until the score is known and may be called from any number of threads at once (it does not take the context's lock).  Calls
 * that arrive together are scored by one kernel launch; a target whose key is already in the device cache is not uploaded again.
 *   max_batch     most requests per launch (<= 0: 64)
 *   max_wait_us   how long the dispatcher waits for company before it launches a partly filled batch
 *   cache_targets code planes kept on every device (2.8 MB each for 1210 x 566); least recently used are replaced.  A device runs several
 *                 independent queues (a third of the host's hardware threads, 2 .. 8; environment CDSGPU_PAIRQ_QUEUES), targets are spread over them by key and each keeps
 *                 cache_targets / queues planes (at least 2 * max_batch)
 *   target_key    the caller's identity of the image (the Java side passes the cache key / System.identityHashCode of the
 *                 ImageArray); equal keys MUST mean equal pixels; 0 = do not cache
 * Scores, ratio and mirrored flag are exactly cds_score_pair_rgb's.  Masks may be ADDED to the mask set while the queue exists (one
 * provider = one mask set + one queue, one algorithm object per mask): the first call that names a new mask pauses the dispatchers
 * between two batches and picks the new masks up.  The mask set must not be destroyed before the queue.  Errors as cds_score_pair_rgb (CDS_ERR_SIZE_MISMATCH for a target of another size). */
typedef struct cds_pairq cds_pairq;
cds_status cds_pairq_create(cds_ctx *ctx, const cds_maskset *ms, int32_t max_batch, int32_t max_wait_us, int32_t cache_targets, cds_pairq **out);
void       cds_pairq_destroy(cds_pairq *q);
cds_status cds_pairq_score(cds_pairq *q, int32_t mask_index, uint64_t target_key, const uint8_t *target_rgb,
                           int32_t target_width, int32_t target_height,
                           int32_t *score_out, double *ratio_out, int32_t *mirrored_out);
/* requests served, kernel launches (batches) and target uploads so far (any pointer may be NULL) */
cds_status cds_pairq_get_stats(const cds_pairq *q, int64_t *requests, int64_t *batches, int64_t *uploads);

/* ---------------------------------------------------------------- shape score ------------------------------------------------------------ */

/* Prepared queries of the shape score.  Replaces createShapeMatchCDSAlgorithmProvider + its per-mask
 * createColorDepthSearchAlgorithm (API/cds/ColorDepthSearchAlgorithmProviderFactory.java:76-127): label clearing,
 * maxFilter(60)/maxFilter(20) high-expression ring, gray>2 query mask.
 * roi_rgb may be NULL.  border must be 0 (CDS_ERR_UNSUPPORTED otherwise; the reference's own unsafeMaxFilter misbehaves
 * for border > kernel radius, SURVEY.md 8a-a8). */
cds_status cds_shape_maskset_create(cds_ctx *ctx, int32_t width, int32_t height, int32_t query_threshold, int32_t border,
                                    int32_t mirror, const cds_rect *rects, int32_t n_rects, const uint8_t *roi_rgb,
                                    cds_shape_maskset **out);
void       cds_shape_maskset_destroy(cds_shape_maskset *sms);
/* qm_size_out / he_size_out (may be NULL): number of set pixels of the query mask and of the high-expression mask
 * (the quantities pinned at 17340 / 70640 by .../cds/Shape2DMatchColorDepthSearchAlgorithmTest.java:53-54). */
cds_status cds_shape_maskset_add_rgb(cds_shape_maskset *sms, const uint8_t *rgb, int32_t n,
                                     int64_t *qm_size_out, int64_t *he_size_out);
int32_t    cds_shape_maskset_size(const cds_shape_maskset *sms);

/* Shape2DMatchColorDepthSearchAlgorithm.calculateMatchingScore for n_pairs (mask, target) pairs
 * (API/cds/Shape2DMatchColorDepthSearchAlgorithm.java:150-245).  Target images come in pair-independent arrays of
 * n_targets images: target_rgb uint8[n_targets][H][W][3], gradient uint16[n_targets][H][W] (gray8 callers widen),
 * zgap_rgb uint8[n_targets][H][W][3] or NULL = derive the zgap image on the device as
 * maxFilter(10)(mask(threshold)(clearLabels(target))) -- what the reference's tests do when no zgap file exists
 * (.../cds/Shape2DMatchColorDepthSearchAlgorithmTest.java:171-174).
 * has_variants uint8[n_targets] (may be NULL = all 1): 0 marks a target whose gradient / zgap supplier is missing;
 * its pairs get gap = high_expr = -1 (:155-158).
 * Outputs per pair: gradientAreaGap, highExpressionArea, mirrored. */
cds_status cds_shape_score_pairs(cds_ctx *ctx, const cds_shape_maskset *sms,
                                 const uint8_t *target_rgb, const uint16_t *gradient, const uint8_t *zgap_rgb,
                                 const uint8_t *has_variants, int64_t n_targets,
                                 const int32_t *pair_mask, const int64_t *pair_target, int64_t n_pairs,
                                 int64_t *gap_out, int64_t *high_expr_out, uint8_t *mirrored_out);

/* The same scoring for targets that are TIFF files in host memory (blob / offsets as in cds_search_stream_tiff): the files are
 * uploaded as stored and decoded on the device, the gradient (and optional zgap) images are passed as pixels as above -- the
 * reference keeps gradients as 16-bit PNG, which it decodes on the JVM (API/imageprocessing/ImageArrayUtils.java:98-121). */
cds_status cds_shape_score_pairs_tiff(cds_ctx *ctx, const cds_shape_maskset *sms, const uint8_t *blob, const int64_t *offsets,
                                      const uint16_t *gradient, const uint8_t *zgap_rgb, const uint8_t *has_variants, int64_t n_targets,
                                      const int32_t *pair_mask, const int64_t *pair_target, int64_t n_pairs,
                                      int64_t *gap_out, int64_t *high_expr_out, uint8_t *mirrored_out);

/* The same scoring with BOTH inputs as files in host memory, the way gradientScores finds them: targets as PackBits / stored RGB
 * TIFF files, gradient images as 16-bit (or 8-bit) grayscale PNG files (png_blob / png_offsets, n_targets + 1 offsets).  The PNG
 * files of a window of targets (up to 2 048) are uploaded as stored and inflated on the device while it works on the previous window
 * (see cds_png_decode_gray16; "device_inflate" 0 inflates them on host threads instead); filters and byte order are undone on the device. */
cds_status cds_shape_score_pairs_files(cds_ctx *ctx, const cds_shape_maskset *sms, const uint8_t *tiff_blob, const int64_t *tiff_offsets,
                                       const uint8_t *png_blob, const int64_t *png_offsets, const uint8_t *zgap_rgb,
                                       const uint8_t *has_variants, int64_t n_targets,
                                       const int32_t *pair_mask, const int64_t *pair_target, int64_t n_pairs,
                                       int64_t *gap_out, int64_t *high_expr_out, uint8_t *mirrored_out);

/* The shape score's single-pair call at scale: a micro-batching scorer with a device-side cache of derived target planes.
 * gradientScores makes one Shape2DMatchColorDepthSearchAlgorithm.calculateMatchingScore(target, variantSuppliers) call per (mask, target)
 * pair (API/cds/Shape2DMatchColorDepthSearchAlgorithm.java:150-245) from a thread pool (TOOLS/CalculateGradientScoresCmd.java:304-312),
 * and the same target recurs across masks.  cds_shape_pairq_score is that call: it blocks its caller until the pair is scored, may be
 * called from any number of threads at once and does not take the context's lock; calls that arrive together are scored by one kernel
 * launch, and a target whose key is already cached is neither uploaded nor derived again.  Returns what cds_shape_score_pairs returns
 * for the same pair, bit for bit.
 *   max_batch, max_wait_us, target_key   as for cds_pairq (several queues per device, environment CDSGPU_PAIRQ_QUEUES); equal keys MUST
 *                 mean equal target, gradient and zgap pixels and the same choice of given or derived zgap image; key 0 = do not cache
 *   cache_targets derived targets kept on every device (at least 2 * max_batch per queue); a slot holds the slice plane, the gradient and
 *                 the signal bitmap: 2 * W * H * 2 + H * bpitch * 4 bytes with bpitch = ceil(W / 32) rounded up to a multiple of 4
 *                 (2.83 MB at 1210 x 566); least recently used are replaced
 *   gradient      uint16[H][W]; NULL = the gradient supplier is missing: (-1, -1, 0) and CDS_OK, no device work (:155-158)
 *   zgap_rgb      uint8[H][W][3] or NULL = derived on the device as in cds_shape_score_pairs
 * Masks may be ADDED to the shape mask set while the queue exists: the first call that names a new mask pauses the dispatchers
 * between two batches and picks the new masks up.  The mask set must not be destroyed before the queue.  CDS_ERR_SIZE_MISMATCH for a
 * target of another size, CDS_ERR_BAD_ARG for a mask index out of range or a NULL target with a gradient. */
typedef struct cds_shape_pairq cds_shape_pairq;
cds_status cds_shape_pairq_create(cds_ctx *ctx, const cds_shape_maskset *sms, int32_t max_batch, int32_t max_wait_us,
                                  int32_t cache_targets, cds_shape_pairq **out);
void       cds_shape_pairq_destroy(cds_shape_pairq *q);
cds_status cds_shape_pairq_score(cds_shape_pairq *q, int32_t mask_index, uint64_t target_key,
                                 const uint8_t *target_rgb, const uint16_t *gradient, const uint8_t *zgap_rgb,
                                 int32_t target_width, int32_t target_height,
                                 int64_t *gap_out, int64_t *high_expr_out, int32_t *mirrored_out);
/* requests served, kernel launches (batches) and target uploads so far (any pointer may be NULL) */
cds_status cds_shape_pairq_get_stats(const cds_shape_pairq *q, int64_t *requests, int64_t *batches, int64_t *uploads);

/* The zgap image alone (f3 in SURVEY.md section 8f): maxFilter(radius)(mask(threshold)(clearLabels(rgb))) for n images. */
cds_status cds_make_zgap(cds_ctx *ctx, const uint8_t *rgb, int64_t n, int32_t width, int32_t height, int32_t threshold,
                         double radius, const cds_rect *rects, int32_t n_rects, uint8_t *zgap_out);

/* ---------------------------------------------------------------- score post-processing -------------------------------------------------- */

/* GradientAreaGapUtils.calculate2DShapeScore (API/cds/GradientAreaGapUtils.java:199-207) and
 * calculateNormalizedScore (:219-235); pure host arithmetic in IEEE double, exposed so bindings do not re-implement it. */
int64_t cds_shape_score_2d(int64_t gradient_area_gap, int64_t high_expression_area);
double  cds_normalized_score(int32_t pixel_match_score, int64_t shape_score, int64_t max_pixel_match, int64_t max_shape_score);
/* CalculateGradientScoresCmd.normalizeScores for one mask's matches (TOOLS/CalculateGradientScoresCmd.java:616-645). */
cds_status cds_normalize_scores(const int32_t *pixel_scores, const int64_t *gaps, const int64_t *high_exprs, int64_t n,
                                float *normalized_out);

/* ---------------------------------------------------------------- match selection (host logic) ------------------------------------------- */

/* ColorMIPProcessUtils.selectBestMatches (TOOLS/cdsprocess/ColorMIPProcessUtils.java:12-34, two nested
 * ItemsHandling.selectTopRankedElements, API/results/ItemsHandling.java:80-109) over the n matches of ONE mask, in the order the
 * reference would hold them: line[i] / sample[i] = dense ids of the target's published name / neuron id (blank names already
 * mapped to "UNKNOWN" by the caller), score[i] = matchingPixels.  line_hash[id] / sample_hash[id] = Java hashCode() of the key
 * string: groups with equal best scores keep java.util.HashMap iteration order, which this call reproduces from the hashes.
 * top_* <= 0 mean "no limit".  selected[] (room for n) receives the indices of the kept matches in the reference's output order:
 * lines by descending best score, inside a line samples by descending best score, inside a sample matches by descending score
 * (ties: input order). */
cds_status cds_select_best_matches(const int32_t *line, const int32_t *sample, const int32_t *score, int64_t n,
                                   const int32_t *line_hash, int32_t n_lines, const int32_t *sample_hash, int32_t n_samples,
                                   int32_t top_lines, int32_t top_samples_per_line, int32_t top_matches_per_sample,
                                   int64_t *selected, int64_t *n_selected);
/* The same selection fused into the searches, on the device (csrc/cds_bestsel.cu): what the reference's two steps keep -- colorDepthSearch
 * writes every pair that passes isMatch, gradientScores reads them back and keeps ColorMIPProcessUtils.selectBestMatches
 * (TOOLS/cdsprocess/ColorMIPProcessUtils.java:12-34, API/results/ItemsHandling.java:80-109) per mask -- without the passing pairs
 * crossing PCIe.  Group keys of the targets are indexed like the targets of the search (library index, or file / image index of a
 * streamed call); every id must lie in [0, n_lines) / [0, n_samples). */
typedef struct cds_target_groups {
    const int32_t *line;          /* [n_targets] dense id of the target's published name (blank -> "UNKNOWN" mapped by the caller) */
    const int32_t *sample;        /* [n_targets] dense id of the neuron id / sample */
    const int32_t *line_hash;     /* [n_lines]   Java String.hashCode() of each line key */
    int32_t        n_lines;
    const int32_t *sample_hash;   /* [n_samples] Java String.hashCode() of each sample key */
    int32_t        n_samples;
} cds_target_groups;

/* Per mask, the pairs of cds_search_matches (same pct_positive_pixels) that cds_select_best_matches keeps, in its output order, masks
 * ascending: the output equals, bit for bit and in the same order, cds_search_matches followed by cds_select_best_matches over each
 * mask's slice (which is already in the reference's encounter order, score descending, then target ascending) with the targets' group
 * ids and hashes.  As a restatement that sorting computes: per (mask, line), best = its highest score and first = the smallest target
 * among its pairs with that score (its first appearance); cap = 16, doubled while the mask's number of distinct lines > 0.75 * cap;
 * bucket = (h ^ (h >>> 16)) & (cap - 1) of the line's hash h.  Lines are ranked by (best desc, bucket asc, first asc) and the first
 * top_lines kept.  Inside a kept line the samples are ranked the same way, cap counting the distinct samples of that line (the
 * reference builds one HashMap per line), and the first top_samples_per_line kept; inside a kept sample the first
 * top_matches_per_sample pairs in encounter order.  Output order: line rank, sample rank, encounter order.  HashMap tree bins are
 * not modelled, as in cds_select_best_matches.
 * top_* <= 0 mean "no limit".  out_* hold `capacity` entries; *out_count receives the number selected; when more are selected than
 * `capacity`, nothing is written, *out_count still tells how many and the call returns CDS_ERR_CAPACITY.  CDS_ERR_SIZE_MISMATCH as
 * cds_search_matches; CDS_ERR_BAD_ARG for a NULL groups or an id outside its range (checked before a device is touched).
 * The passing pairs are kept on the devices, at most "best_list_bytes" per device (cds_ctx_set_option).  When a list fills and
 * top_matches_per_sample > 0 it is compacted to the first top_matches_per_sample pairs of every (mask, line, sample), which changes no
 * selection (every present sample keeps its best pair, so best / first of lines and samples and the numbers of distinct lines and
 * samples stay); when it still does not fit, or top_matches_per_sample <= 0, the call returns CDS_ERR_CAPACITY naming the bytes needed.
 * On a context of several devices the lists are moved to the first device (peer copies, staged through pinned host memory where
 * peer access is missing) and selected there.  Only the selected pairs and their count cross to the host (cds_search_stats.d2h_bytes).
 * One process per GPU (colormipsearch_b200/sharding.py) does NOT give an exact selection -- a mask's pairs would have to meet from
 * every rank; use one context over the devices instead. */
cds_status cds_search_best_matches(cds_ctx *ctx, const cds_maskset *ms, cds_library *lib, const cds_target_groups *groups,
                                   double pct_positive_pixels, int32_t top_lines, int32_t top_samples_per_line, int32_t top_matches_per_sample,
                                   int64_t capacity, int32_t *out_mask, int64_t *out_target, int32_t *out_score, uint8_t *out_mirrored,
                                   int64_t *out_count);
/* The same over TIFF files / RGB images in host memory (targets as in cds_search_stream_matches_tiff / _rgb). */
cds_status cds_search_stream_best_matches_tiff(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *blob, const int64_t *offsets,
                                               int64_t n_targets, const cds_target_groups *groups, double pct_positive_pixels,
                                               int32_t top_lines, int32_t top_samples_per_line, int32_t top_matches_per_sample,
                                               int64_t capacity, int32_t *out_mask, int64_t *out_target, int32_t *out_score,
                                               uint8_t *out_mirrored, int64_t *out_count);
cds_status cds_search_stream_best_matches_rgb(cds_ctx *ctx, const cds_maskset *ms, const uint8_t *targets_rgb, int64_t n_targets,
                                              const cds_target_groups *groups, double pct_positive_pixels,
                                              int32_t top_lines, int32_t top_samples_per_line, int32_t top_matches_per_sample,
                                              int64_t capacity, int32_t *out_mask, int64_t *out_target, int32_t *out_score,
                                              uint8_t *out_mirrored, int64_t *out_count);
/* Test hook: the device selection alone, on the context's first device, over a caller-given list of one or more masks' passing pairs
 * sorted by (mask, score desc, target asc) (CDS_ERR_BAD_ARG otherwise); groups are indexed by target.  selected[] (room for n)
 * receives indices into that list in output order; *n_selected their number. */
cds_status cds_debug_select_best_matches_device(cds_ctx *ctx, const int32_t *mask, const int64_t *target, const int32_t *score,
                                                const uint8_t *mirrored, int64_t n, const cds_target_groups *groups, int32_t top_lines,
                                                int32_t top_samples_per_line, int32_t top_matches_per_sample, int64_t *selected,
                                                int64_t *n_selected);
/* java.lang.String.hashCode() of an ASCII string (helper for non-Java callers of cds_select_best_matches). */
int32_t cds_java_string_hash(const char *ascii);

/* ---------------------------------------------------------------- synthetic inputs + instrumentation ------------------------------------- */

/* Deterministic synthetic images, identical bit for bit on host and device (bench.py, scale tests).
 * kind: 0 = EM-like mask, 1 = LM-like target.  Writes n RGB images for indices first_index.. into rgb_out (host).
 * on_device != 0 generates with the CUDA generator and copies back; 0 uses the host build of the same generator. */
cds_status cds_synth_rgb(cds_ctx *ctx, int32_t kind, uint64_t seed, int64_t first_index, int64_t n,
                         int32_t width, int32_t height, int32_t on_device, uint8_t *rgb_out);
/* gradient image (gray16) of synthetic target `index`: capped distance to the nearest generated neurite. */
cds_status cds_synth_gradient(cds_ctx *ctx, uint64_t seed, int64_t first_index, int64_t n,
                              int32_t width, int32_t height, int32_t on_device, uint16_t *grad_out);

/* Counters of the last search on this ctx (bench.py reads them): kernel launches, device milliseconds of the
 * dominant kernel summed over launches (CUDA events on the launch stream, max over devices), comparisons done. */
typedef struct cds_search_stats {
    int64_t kernel_launches;
    int64_t match_kernel_launches;
    double  match_kernel_ms;
    double  total_device_ms;
    int64_t comparisons;
    int64_t h2d_bytes;
    int64_t d2h_bytes;
    int64_t match_kernel;        /* which match kernel the last launch used: 1 candidate, 2 band, 3 gather */
    int64_t chunked;             /* 1 when the search walked its targets in chunks (streamed targets, or occupancy bitmaps built per chunk) */
    int64_t host_inflate_fallbacks;   /* cds_shape_score_pairs_files: gradient PNG streams the device's inflate refused and zlib read on the host */
} cds_search_stats;
cds_status cds_get_last_stats(const cds_ctx *ctx, cds_search_stats *out);

/* Test hooks (tests/ only): the encoded form of colours and the per-class match intervals, so that the integer
 * predicate used on the device can be checked exhaustively against the oracle's double arithmetic. */
cds_status cds_debug_encode_colors(cds_ctx *ctx, const uint8_t *rgb, int64_t n, int32_t data_threshold, uint32_t *codes_out);
cds_status cds_debug_class_intervals(double z_tolerance, int32_t sector, int32_t rank,
                                     uint32_t *lo1, uint32_t *len1, uint32_t *lo2, uint32_t *len2);
/* n TIFF files (blob / offsets as in cds_search_stream_tiff) -> the code words a streaming search builds from them, uint32[n][H][W]
 * (cds_common.h), and optionally the per-sector "can match" bits uint32[n][H][6][ceil32(W) rounded up to 4 words]; fused != 0 runs
 * the fused strip -> code-word kernel, 0 the decode + encode pair.  Lets tests compare the two ingest paths word for word. */
cds_status cds_debug_tiff_codes(cds_ctx *ctx, const uint8_t *blob, const int64_t *offsets, int64_t n, int32_t width, int32_t height,
                                int32_t data_threshold, int32_t fused, uint32_t *codes_out, uint32_t *valid_out);
/* Drives cds_pairq_score from n_threads native threads over a list of pairs, the way the reference's thread pool drives
 * calculateMatchingScore: thread-safety tests and the throughput number of the single-pair entry point (bench.py). */
/* Test hook: per-sector valid bits [n][height][6][vp] (vp = ((width + 31) / 32 rounded up to a multiple of 4) words per row and sector,
 * bit x % 32 of word x / 32) -> the occupancy tile rows built from them for xy_shift 0 / 2 / 4, [n][(height + 3) / 4][row pitch] with
 * row pitch = 7 * tp + nz words (tp = (width + 7) / 8 rounded up to a multiple of 4; nz = ((6 * tp + 31) / 32 rounded up to a multiple of
 * 4): six sector rows of 8 x 4 tile words, their OR row, one "non-empty" bit per sector tile word.  The words between the rows are all written. */
cds_status cds_debug_occupancy(cds_ctx *ctx, const uint32_t *valid, int64_t n, int32_t width, int32_t height, int32_t xy_shift,
                               uint32_t *occ_out);
/* Test hook: the rank-band bytes that a search with data_threshold and xy_shift (0, 2, 4) finds in the library's resident occupancy
 * (baking the library at data_threshold and building the occupancy first, as such a search does): uint8[size][(height + 3) / 4][6 * tp],
 * tp as above; byte [t][ty][sector * tp + tx] has bit b set when a pixel of target t in that colour sector, inside the image, above
 * data_threshold and in [8 tx - S, 8 tx + 7 + S] x [4 ty - S, 4 ty + 3 + S] (S = xy_shift) has rank band b = rank * 8 / 19820.
 * CDS_ERR_UNSUPPORTED when the library has no room for resident occupancy and builds it per chunk. */
cds_status cds_debug_library_bands(cds_library *lib, int32_t data_threshold, int32_t xy_shift, uint8_t *bands_out);
/* Test hook (no device needed): how the candidate kernel would run at this image size, xy_shift (0, 2, 4) and palette size
 * (palette_entries = the largest palette of the launch's mask groups plus one idle entry, 1..2048; ignored when wide != 0, since wide
 * word lists read no palette): consumer warps per block, image rows per band, band stages in flight and dynamic shared memory in bytes.
 * All four are 0 when no configuration fits. */
cds_status cds_debug_cand_config(int32_t width, int32_t height, int32_t xy_shift, int32_t palette_entries, int32_t wide,
                                 int32_t *warps, int32_t *rows_per_band, int32_t *stages, int64_t *smem_bytes);
/* Test hook (no device needed): the chunk plan of the streaming searches over host targets -- entry i = (device, first target, count).
 * offsets == NULL: pixels (equal chunks of `chunk` targets, round-robin over the devices); otherwise the files' offsets [n_targets + 1]:
 * the first chunks of every device are 256, 512, ... files, what is left after the ramp is cut into equal chunks of at most `chunk`, and a
 * chunk ends where its files would exceed byte_cap.  *n_out = entries; CDS_ERR_CAPACITY when capacity is too small. */
cds_status cds_debug_stream_plan(int32_t n_devices, int64_t n_targets, int64_t chunk, const int64_t *offsets, int64_t byte_cap,
                                 int64_t capacity, int32_t *dev_out, int64_t *first_out, int64_t *count_out, int64_t *n_out);
cds_status cds_debug_pairq_drive(cds_pairq *q, const uint8_t *targets_rgb, int64_t n_targets, const uint64_t *keys,
                                 const int32_t *pair_mask, const int64_t *pair_target, int64_t n_pairs, int32_t n_threads,
                                 int32_t *scores_out, uint8_t *mirrored_out, double *seconds_out);
/* Drives cds_shape_pairq_score from n_threads native threads over a list of pairs, like cds_debug_pairq_drive: target t is
 * targets_rgb[t], gradients[t] and zgaps_rgb[t] (zgaps_rgb may be NULL: derived) with key keys[t] (keys may be NULL: 0).
 * seconds_out = wall clock of the whole run. */
cds_status cds_debug_shape_pairq_drive(cds_shape_pairq *q, const uint8_t *targets_rgb, const uint16_t *gradients,
                                       const uint8_t *zgaps_rgb, int64_t n_targets, const uint64_t *keys,
                                       const int32_t *pair_mask, const int64_t *pair_target, int64_t n_pairs, int32_t n_threads,
                                       int64_t *gap_out, int64_t *high_expr_out, uint8_t *mirrored_out, double *seconds_out);
/* Slice numbers (1..256, 0 = black) of n RGB colours as the shape path computes them on the device -- a table built per device
 * with the double arithmetic of GradientAreaGapUtils.findSliceNumberInLUT (API/cds/GradientAreaGapUtils.java:18-197) -- so that the
 * table can be checked against the oracle over all 2^24 colours. */
cds_status cds_debug_slice_numbers(cds_ctx *ctx, const uint8_t *rgb, int64_t n, uint16_t *slices_out);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* CDSGPU_H */

package org.janelia.colormipsearch.cds.gpu;

import java.lang.foreign.Arena;
import java.lang.foreign.FunctionDescriptor;
import java.lang.foreign.Linker;
import java.lang.foreign.MemoryLayout;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.StructLayout;
import java.lang.foreign.SymbolLookup;
import java.lang.foreign.ValueLayout;
import java.lang.invoke.MethodHandle;

import static java.lang.foreign.ValueLayout.ADDRESS;
import static java.lang.foreign.ValueLayout.JAVA_DOUBLE;
import static java.lang.foreign.ValueLayout.JAVA_INT;
import static java.lang.foreign.ValueLayout.JAVA_LONG;

/**
 * Panama FFM (JDK 22+) binding of libcdsgpu.so, the C ABI declared in include/cdsgpu.h.
 * One downcall handle per exported function; no generated headers, no JNI code.
 *
 * UNVERIFIED: written against the JDK 22 java.lang.foreign API; the build image of the GPU library has no JDK, so this
 * file has not been compiled.  The same ABI is exercised from C++ (colormipsearch_b200/host/cds_host.hpp) and from Python
 * ctypes (colormipsearch_b200/capi.py) by the test suite.
 */
public final class CdsGpu {
    public static final int CDS_OK = 0, CDS_ERR_BAD_ARG = 1, CDS_ERR_SIZE_MISMATCH = 2, CDS_ERR_CAPACITY = 6, CDS_ERR_UNSUPPORTED = 7;
    public static final int CDS_MAX_RECTS = 8;

    /** cds_rect {int32 x0, y0, x1, y1} */
    static final StructLayout RECT = MemoryLayout.structLayout(JAVA_INT.withName("x0"), JAVA_INT.withName("y0"), JAVA_INT.withName("x1"), JAVA_INT.withName("y1"));
    /** cds_pixparams: int32 mask_threshold, int32 data_threshold, double z_tolerance, int32 xy_shift, mirror, n_rects, cds_rect rects[8] (+4 bytes tail padding) */
    static final StructLayout PIXPARAMS = MemoryLayout.structLayout(
            JAVA_INT.withName("mask_threshold"), JAVA_INT.withName("data_threshold"), JAVA_DOUBLE.withName("z_tolerance"),
            JAVA_INT.withName("xy_shift"), JAVA_INT.withName("mirror"), JAVA_INT.withName("n_rects"),
            MemoryLayout.sequenceLayout(CDS_MAX_RECTS, RECT).withName("rects"), MemoryLayout.paddingLayout(4));

    private static final Linker LINKER = Linker.nativeLinker();
    private static final SymbolLookup LIB = SymbolLookup.libraryLookup(
            System.getProperty("cdsgpu.library", "libcdsgpu.so"), Arena.global());

    private static MethodHandle h(String name, FunctionDescriptor fd) {
        return LINKER.downcallHandle(LIB.find(name).orElseThrow(() -> new UnsatisfiedLinkError(name)), fd);
    }

    public static final MethodHandle ctxCreate = h("cds_ctx_create", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS));
    public static final MethodHandle ctxDestroy = h("cds_ctx_destroy", FunctionDescriptor.ofVoid(ADDRESS));
    public static final MethodHandle lastError = h("cds_last_error", FunctionDescriptor.of(ADDRESS, ADDRESS));
    public static final MethodHandle hostAlloc = h("cds_host_alloc", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS));
    public static final MethodHandle hostFree = h("cds_host_free", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    public static final MethodHandle libraryCreate = h("cds_library_create", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_LONG, ADDRESS));
    public static final MethodHandle libraryDestroy = h("cds_library_destroy", FunctionDescriptor.ofVoid(ADDRESS));
    public static final MethodHandle libraryAddRgb = h("cds_library_add_rgb", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
    public static final MethodHandle masksetCreate = h("cds_maskset_create", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS, ADDRESS));
    public static final MethodHandle masksetDestroy = h("cds_maskset_destroy", FunctionDescriptor.ofVoid(ADDRESS));
    public static final MethodHandle masksetAddRgb = h("cds_maskset_add_rgb", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS));
    public static final MethodHandle searchTopk = h("cds_search_topk", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, JAVA_DOUBLE, ADDRESS, ADDRESS, ADDRESS, ADDRESS));
    public static final MethodHandle searchStream = h("cds_search_stream_rgb", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_DOUBLE, ADDRESS, ADDRESS, ADDRESS, ADDRESS));
    public static final MethodHandle searchStreamMatches = h("cds_search_stream_matches_rgb", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_DOUBLE, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS));
    // image ingest: TIFF files as stored, decoded on the device (include/cdsgpu.h, "image ingest")
    public static final MethodHandle masksetAddTiff = h("cds_maskset_add_tiff", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, ADDRESS));
    public static final MethodHandle libraryAddTiff = h("cds_library_add_tiff", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
    public static final MethodHandle searchStreamTiff = h("cds_search_stream_tiff", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_DOUBLE, ADDRESS, ADDRESS, ADDRESS, ADDRESS));
    public static final MethodHandle searchStreamMatchesTiff = h("cds_search_stream_matches_tiff", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_DOUBLE, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS));
    // cds_search_best_matches(ctx, maskset, library, const cds_target_groups *groups, pct, topLines, topSamplesPerLine, topMatchesPerSample,
    //                         capacity, outMask, outTarget, outScore, outMirrored, outCount): selectBestMatches fused into the search, on the
    // device.  cds_target_groups = {int *line, int *sample, int *lineHash, int nLines, int *sampleHash, int nSamples} (natural C layout, 48 bytes).
    public static final MethodHandle searchBestMatches = h("cds_search_best_matches", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_DOUBLE, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS));
    public static final MethodHandle shapeScorePairsTiff = h("cds_shape_score_pairs_tiff", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS));
    public static final MethodHandle tiffProbe = h("cds_tiff_probe", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS));
    // the single-pair call behind a micro-batching queue with a device-side target cache (include/cdsgpu.h, cds_pairq_*)
    public static final MethodHandle pairqCreate = h("cds_pairq_create", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS));
    public static final MethodHandle pairqDestroy = h("cds_pairq_destroy", FunctionDescriptor.ofVoid(ADDRESS));
    public static final MethodHandle pairqScore = h("cds_pairq_score", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_LONG, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    // gradient images as PNG files, targets as TIFF files
    public static final MethodHandle shapeScorePairsFiles = h("cds_shape_score_pairs_files", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS));
    public static final MethodHandle tiffToPackbits = h("cds_tiff_to_packbits", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS, JAVA_LONG, ADDRESS));
    public static final MethodHandle tiffEncodeBound = h("cds_tiff_encode_bound", FunctionDescriptor.of(JAVA_LONG, JAVA_INT, JAVA_INT, JAVA_INT));
    public static final MethodHandle scorePairRgb = h("cds_score_pair_rgb", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    public static final MethodHandle shapeMasksetCreate = h("cds_shape_maskset_create", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS));
    public static final MethodHandle shapeMasksetDestroy = h("cds_shape_maskset_destroy", FunctionDescriptor.ofVoid(ADDRESS));
    public static final MethodHandle shapeMasksetAddRgb = h("cds_shape_maskset_add_rgb", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS));
    public static final MethodHandle shapeScorePairs = h("cds_shape_score_pairs", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS));

    /** One context per JVM: the lifetime of a command run (colorDepthSearch / gradientScores). */
    private static volatile MemorySegment CTX;

    public static MemorySegment context() {
        MemorySegment c = CTX;
        if (c == null) {
            synchronized (CdsGpu.class) {
                if (CTX == null) {
                    try (Arena a = Arena.ofConfined()) {
                        MemorySegment out = a.allocate(ADDRESS);
                        int nDev = Integer.getInteger("cdsgpu.devices", 0);   // 0 = every visible GPU
                        int st = (int) ctxCreate.invokeExact(MemorySegment.NULL, nDev, out);
                        if (st != CDS_OK) throw new IllegalStateException(errorMessage(MemorySegment.NULL));
                        CTX = out.get(ADDRESS, 0);
                    } catch (RuntimeException e) {
                        throw e;
                    } catch (Throwable t) {
                        throw new IllegalStateException(t);
                    }
                }
                c = CTX;
            }
        }
        return c;
    }

    static String errorMessage(MemorySegment ctx) {
        try {
            MemorySegment s = (MemorySegment) lastError.invokeExact(ctx);
            return s.reinterpret(Long.MAX_VALUE).getString(0);
        } catch (Throwable t) {
            return "cds_last_error failed: " + t;
        }
    }

    /** Error convention of the C ABI (include/cdsgpu.h): bad argument / size mismatch are the reference's IllegalArgumentException sites. */
    public static void check(int status) {
        if (status == CDS_OK) return;
        String msg = errorMessage(context());
        if (status == CDS_ERR_BAD_ARG || status == CDS_ERR_SIZE_MISMATCH) throw new IllegalArgumentException(msg);
        throw new IllegalStateException(msg);
    }

    /** Fills a cds_pixparams in `arena`. */
    public static MemorySegment pixParams(Arena arena, int maskThreshold, int dataThreshold, double zTolerance, int xyShift, boolean mirror, int[][] rects) {
        MemorySegment p = arena.allocate(PIXPARAMS);
        p.set(JAVA_INT, 0, maskThreshold);
        p.set(JAVA_INT, 4, dataThreshold);
        p.set(JAVA_DOUBLE, 8, zTolerance);
        p.set(JAVA_INT, 16, xyShift);
        p.set(JAVA_INT, 20, mirror ? 1 : 0);
        p.set(JAVA_INT, 24, rects.length);
        for (int i = 0; i < rects.length; i++)
            for (int k = 0; k < 4; k++) p.set(JAVA_INT, 28 + 16L * i + 4L * k, rects[i][k]);
        return p;
    }

    public static MemorySegment copyBytes(Arena arena, byte[] a) {
        MemorySegment s = arena.allocate(a.length);
        MemorySegment.copy(a, 0, s, ValueLayout.JAVA_BYTE, 0, a.length);
        return s;
    }

    private CdsGpu() {}
}

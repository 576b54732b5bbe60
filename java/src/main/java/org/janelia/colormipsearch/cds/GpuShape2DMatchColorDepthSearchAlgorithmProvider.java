package org.janelia.colormipsearch.cds;

import java.lang.foreign.Arena;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.ValueLayout;
import java.util.EnumSet;
import java.util.Map;
import java.util.Set;
import java.util.function.Supplier;

import javax.annotation.Nonnull;

import org.janelia.colormipsearch.cds.gpu.CdsGpu;
import org.janelia.colormipsearch.imageprocessing.ImageArray;
import org.janelia.colormipsearch.imageprocessing.ImageArrayAccess;
import org.janelia.colormipsearch.imageprocessing.ImageRegionDefinition;
import org.janelia.colormipsearch.model.ComputeFileType;

/**
 * Drop-in for createShapeMatchCDSAlgorithmProvider (ColorDepthSearchAlgorithmProviderFactory.java:76-127).  Lives in package
 * org.janelia.colormipsearch.cds because ShapeMatchScore's constructors are package-private (ShapeMatchScore.java:12,20).
 *
 * Every calculateMatchingScore is one blocking cds_shape_pairq_score call.  The calls of gradientScores' pool threads
 * (CalculateGradientScoresCmd.java:304-312) meet in the library's micro-batching queue and are scored by one kernel launch per batch;
 * a target that was scored before is found in the device-side cache of derived planes by its identity (the same key as the pixel
 * provider's), so it is uploaded and derived once.  All algorithms of one parameter set share ONE native shape mask set and ONE queue
 * (masks are appended as algorithms are created).
 *
 * UNVERIFIED (no JDK in the build image of the GPU library).
 */
public class GpuShape2DMatchColorDepthSearchAlgorithmProvider implements ColorDepthSearchAlgorithmProvider<ShapeMatchScore> {
    private final ColorDepthSearchParams defaults = new ColorDepthSearchParams();
    private final ImageArray<?> roiMask;
    private final ImageRegionDefinition excludedRegions;

    public GpuShape2DMatchColorDepthSearchAlgorithmProvider(boolean mirrorMask, ImageArray<?> roiMaskImageArray, ImageRegionDefinition excludedRegions) {
        defaults.setParam("mirrorMask", mirrorMask);
        this.roiMask = roiMaskImageArray;
        this.excludedRegions = excludedRegions;
    }

    @Override public ColorDepthSearchParams getDefaultCDSParams() { return defaults; }

    /** One native shape mask set + pair queue per (image size, query threshold, border, mirror, excluded rectangles). */
    private static final class Shared {
        MemorySegment maskSet, queue;
        int nMasks;
    }
    private final Map<String, Shared> shared = new java.util.HashMap<>();

    private synchronized int addMask(String key, ImageArray<?> queryImage, int queryThreshold, int border, boolean mirror, int[][] rects,
                                     Shared[] out, int[] sizeOut) {
        Shared sh = shared.get(key);
        try (Arena a = Arena.ofConfined()) {
            MemorySegment o = a.allocate(ValueLayout.ADDRESS), qm = a.allocate(ValueLayout.JAVA_LONG), he = a.allocate(ValueLayout.JAVA_LONG);
            if (sh == null) {
                sh = new Shared();
                MemorySegment r = a.allocate(16L * Math.max(rects.length, 1));
                for (int i = 0; i < rects.length; i++) for (int k = 0; k < 4; k++) r.set(ValueLayout.JAVA_INT, 16L * i + 4L * k, rects[i][k]);
                MemorySegment roiSeg = roiMask == null ? MemorySegment.NULL : CdsGpu.copyBytes(a, ImageArrayAccess.rgbBytes(roiMask));
                CdsGpu.check((int) CdsGpu.shapeMasksetCreate.invokeExact(CdsGpu.context(), queryImage.getWidth(), queryImage.getHeight(), queryThreshold, border,
                        mirror ? 1 : 0, r, rects.length, roiSeg, o));
                sh.maskSet = o.get(ValueLayout.ADDRESS, 0);
                shared.put(key, sh);
            }
            CdsGpu.check((int) CdsGpu.shapeMasksetAddRgb.invokeExact(sh.maskSet, CdsGpu.copyBytes(a, ImageArrayAccess.rgbBytes(queryImage)), 1, qm, he));
            sizeOut[0] = (int) qm.get(ValueLayout.JAVA_LONG, 0);
            if (sh.queue == null) {
                // max batch 256, wait at most 60 us for company, 1024 derived targets per device (2.9 GB for 1210 x 566)
                CdsGpu.check((int) CdsGpu.shapePairqCreate.invokeExact(CdsGpu.context(), sh.maskSet, 256, 60, Integer.getInteger("cdsgpu.cachedShapeTargets", 1024), o));
                sh.queue = o.get(ValueLayout.ADDRESS, 0);
            }
            out[0] = sh;
            return sh.nMasks++;
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
    }

    @Override
    public ColorDepthSearchAlgorithm<ShapeMatchScore> createColorDepthSearchAlgorithm(ImageArray<?> queryImage, int queryThreshold,
                                                                                      int queryBorderSize, ColorDepthSearchParams cdsParams) {
        boolean mirror = cdsParams.getBoolParam("mirrorMask", defaults.getBoolParam("mirrorMask", false));
        int[][] rects = GpuPixelMatchColorDepthSearchAlgorithmProvider.rectanglesOf(excludedRegions, queryImage);
        String key = queryImage.getWidth() + "x" + queryImage.getHeight() + ":" + queryThreshold + ":" + queryBorderSize + ":" + mirror
                + ":" + java.util.Arrays.deepToString(rects);
        Shared[] sh = new Shared[1];
        int[] size = new int[1];
        int index = addMask(key, queryImage, queryThreshold, queryBorderSize, mirror, rects, sh, size);
        return new Algorithm(queryImage, sh[0].queue, index, size[0]);
    }

    static final class Algorithm implements ColorDepthSearchAlgorithm<ShapeMatchScore> {
        private static final Set<ComputeFileType> REQUIRED = EnumSet.of(ComputeFileType.GradientImage, ComputeFileType.ZGapImage);
        private final ImageArray<?> queryImage;
        private final transient MemorySegment queue;   // native handle: not serialisable, Spark mode is unsupported on this provider
        private final int maskIndex, querySize;

        Algorithm(ImageArray<?> queryImage, MemorySegment queue, int maskIndex, int querySize) {
            this.queryImage = queryImage; this.queue = queue; this.maskIndex = maskIndex; this.querySize = querySize;
        }

        @Override public ImageArray<?> getQueryImage() { return queryImage; }
        @Override public int getQuerySize() { return querySize; }
        @Override public int getQueryFirstPixelIndex() { return 0; }
        @Override public int getQueryLastPixelIndex() { return queryImage.getPixelCount() - 1; }
        @Override public Set<ComputeFileType> getRequiredTargetVariantTypes() { return REQUIRED; }

        /** Thread-safe and re-entrant: cds_shape_pairq_score takes no context-wide lock; calls that arrive together share a kernel launch. */
        @Override
        public ShapeMatchScore calculateMatchingScore(@Nonnull ImageArray<?> target, Map<ComputeFileType, Supplier<ImageArray<?>>> variants) {
            ImageArray<?> grad = fetch(variants, ComputeFileType.GradientImage), zgap = fetch(variants, ComputeFileType.ZGapImage);
            if (grad == null || zgap == null) return new ShapeMatchScore(-1, -1, -1, false);   // Shape2DMatch...:155-158
            try (Arena a = Arena.ofConfined()) {
                int n = target.getPixelCount();
                MemorySegment g16 = a.allocate(2L * n, 2);
                if (ImageArrayAccess.isGray16(grad)) MemorySegment.copy(ImageArrayAccess.gray16(grad), 0, g16, ValueLayout.JAVA_SHORT, 0, n);
                else { byte[] g8 = ImageArrayAccess.gray8(grad); for (int i = 0; i < n; i++) g16.set(ValueLayout.JAVA_SHORT, 2L * i, (short) (g8[i] & 0xFF)); }
                MemorySegment gap = a.allocate(ValueLayout.JAVA_LONG), he = a.allocate(ValueLayout.JAVA_LONG), mir = a.allocate(ValueLayout.JAVA_INT);
                // the key is the target ImageArray's identity: its gradient and zgap images come with it
                CdsGpu.check((int) CdsGpu.shapePairqScore.invokeExact(queue, maskIndex, GpuPixelMatchColorDepthSearchAlgorithmProvider.targetKey(target),
                        CdsGpu.copyBytes(a, ImageArrayAccess.rgbBytes(target)), g16, CdsGpu.copyBytes(a, ImageArrayAccess.rgbBytes(zgap)),
                        target.getWidth(), target.getHeight(), gap, he, mir));
                return new ShapeMatchScore(gap.get(ValueLayout.JAVA_LONG, 0), he.get(ValueLayout.JAVA_LONG, 0), -1, mir.get(ValueLayout.JAVA_INT, 0) != 0);
            } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
        }

        private static ImageArray<?> fetch(Map<ComputeFileType, Supplier<ImageArray<?>>> v, ComputeFileType t) {
            Supplier<ImageArray<?>> s = v == null ? null : v.get(t);
            return s == null ? null : s.get();
        }
    }
}

package com.android.nQuant.b200;

import java.lang.foreign.Arena;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.ValueLayout;

/**
 * Drop-in for the quantizer core of com.android.nQuant.PnnQuantizer (reference
 * nQuant.master/src/main/java/com/android/nQuant/PnnQuantizer.java): same constructor role, same
 * convert(nMaxColors, dither) and hasAlpha(), over an ARGB int[] in place of android.graphics.Bitmap.
 * All arithmetic runs in libnquant_b200.so (CUDA, sm_100a); there is no Java fallback.
 *
 * Differences from the reference, all forced by the boundary:
 *  - the constructor takes the pixels the reference obtains with Bitmap.getPixels (PnnQuantizer.java:39-44);
 *  - convert returns the int[] the reference hands to Bitmap.createBitmap (PnnQuantizer.java:455);
 *  - the protected overridables (getQuanFn, pnnquan, nearestColorIndex, closestColorIndex, dither) do
 *    not exist here: a per-pixel Java callback cannot run inside a CUDA kernel.
 *
 * NOT COMPILED IN THIS REPOSITORY'S BUILD IMAGE (no JDK); see INTEGRATION.md.
 */
public class PnnQuantizer implements AutoCloseable {
	protected final int[] pixels;
	protected final int width, height;
	protected final int device;
	protected final long rngSeed;
	protected boolean hasAlpha;
	protected int[] palette = new int[0];

	public PnnQuantizer(int[] argb, int width, int height) {
		this(argb, width, height, 0, 0L);
	}

	/** @param rngSeed seed of the java.util.Random behind PnnLABQuantizer.closestColorIndex
	 *                 (unseeded and static in the reference, PnnLABQuantizer.java:22,467). */
	public PnnQuantizer(int[] argb, int width, int height, int device, long rngSeed) {
		if (argb.length != width * height)
			throw new IllegalArgumentException("argb must hold width*height pixels");
		this.pixels = argb.clone();     // the reference keeps a private copy too (PnnQuantizer.java:42-43)
		this.width = width;
		this.height = height;
		this.device = device;
		this.rngSeed = rngSeed;
		NQuantNative.context(device);   // fails here, like the reference's constructor would on a bad file, not in convert
	}

	protected int kind() {
		return NQuantNative.NQ_KIND_PNN;
	}

	/** Bitmap convert(int nMaxColors, boolean dither) throws Exception (PnnQuantizer.java:409). */
	public int[] convert(int nMaxColors, boolean dither) throws Exception {
		try (Arena arena = Arena.ofConfined()) {
			final long n = (long) width * height;
			MemorySegment in = arena.allocateFrom(ValueLayout.JAVA_INT, pixels);
			MemorySegment out = arena.allocate(ValueLayout.JAVA_INT, n);
			MemorySegment pal = arena.allocate(ValueLayout.JAVA_INT, 256);
			MemorySegment plen = arena.allocate(ValueLayout.JAVA_INT);
			MemorySegment alpha = arena.allocate(ValueLayout.JAVA_INT);
			int rc;
			try {
				rc = (int) NQuantNative.nq_convert.invokeExact(NQuantNative.context(device), kind(), in, width, height, nMaxColors,
					dither ? 1 : 0, rngSeed, out, pal, plen, alpha);
			} catch (Throwable t) {
				throw new Exception(t);
			}
			if (rc != 0)
				throw new Exception("nq_convert failed (" + rc + "): " + NQuantNative.lastError());
			hasAlpha = alpha.get(ValueLayout.JAVA_INT, 0) != 0;
			palette = pal.asSlice(0, 4L * plen.get(ValueLayout.JAVA_INT, 0)).toArray(ValueLayout.JAVA_INT);
			return out.toArray(ValueLayout.JAVA_INT);
		}
	}

	/**
	 * convert() as palette indices, one byte per pixel, computed on the GPU (nq_convert_ragged_indexed): what an indexed
	 * format (PNG8, GIF, a palette texture) stores. getPalette()[index & 0xFF] is the colour convert() returns for the pixel
	 * (the lowest index of that colour). The colours themselves are not copied back. Sets getPalette() and hasAlpha() like
	 * convert().
	 */
	public byte[] convertIndexed(int nMaxColors, boolean dither) throws Exception {
		try (Arena arena = Arena.ofConfined()) {
			final long n = (long) width * height;
			MemorySegment in = arena.allocate(ValueLayout.ADDRESS);
			in.set(ValueLayout.ADDRESS, 0, arena.allocateFrom(ValueLayout.JAVA_INT, pixels));
			MemorySegment idx = arena.allocate(n);
			MemorySegment idxs = arena.allocate(ValueLayout.ADDRESS);
			idxs.set(ValueLayout.ADDRESS, 0, idx);
			MemorySegment w = arena.allocateFrom(ValueLayout.JAVA_INT, width);
			MemorySegment h = arena.allocateFrom(ValueLayout.JAVA_INT, height);
			MemorySegment seed = arena.allocateFrom(ValueLayout.JAVA_LONG, rngSeed);
			MemorySegment pal = arena.allocate(ValueLayout.JAVA_INT, 256);
			MemorySegment plen = arena.allocate(ValueLayout.JAVA_INT);
			MemorySegment alpha = arena.allocate(ValueLayout.JAVA_INT);
			int rc;
			try {
				rc = (int) NQuantNative.nq_convert_ragged_indexed.invokeExact(NQuantNative.context(device), kind(), in, w, h, 1, nMaxColors,
					dither ? 1 : 0, seed, idxs, MemorySegment.NULL, pal, plen, alpha);
			} catch (Throwable t) {
				throw new Exception(t);
			}
			if (rc != 0)
				throw new Exception("nq_convert_ragged_indexed failed (" + rc + "): " + NQuantNative.lastError());
			hasAlpha = alpha.get(ValueLayout.JAVA_INT, 0) != 0;
			palette = pal.asSlice(0, 4L * plen.get(ValueLayout.JAVA_INT, 0)).toArray(ValueLayout.JAVA_INT);
			return idx.toArray(ValueLayout.JAVA_BYTE);
		}
	}

	/**
	 * convert() with the palette replaced by the caller's (nq_remap_ragged): the alpha scan and the histogram's scalars as
	 * convert(nMaxColors, dither) computes them, no merge loop, then the dither to {@code palette} (1..256 colours). Remapping
	 * to the palette convert() returned, with the same nMaxColors and seed, returns convert()'s output. Sets hasAlpha() and
	 * makes getPalette() return {@code palette}.
	 */
	public int[] remap(int[] palette, int nMaxColors, boolean dither) throws Exception {
		if (palette.length < 1 || palette.length > 256)
			throw new IllegalArgumentException("palette must hold 1..256 colours");
		try (Arena arena = Arena.ofConfined()) {
			final long n = (long) width * height;
			MemorySegment in = arena.allocate(ValueLayout.ADDRESS);
			in.set(ValueLayout.ADDRESS, 0, arena.allocateFrom(ValueLayout.JAVA_INT, pixels));
			MemorySegment out = arena.allocate(ValueLayout.JAVA_INT, n);
			MemorySegment outs = arena.allocate(ValueLayout.ADDRESS);
			outs.set(ValueLayout.ADDRESS, 0, out);
			MemorySegment w = arena.allocateFrom(ValueLayout.JAVA_INT, width);
			MemorySegment h = arena.allocateFrom(ValueLayout.JAVA_INT, height);
			MemorySegment seed = arena.allocateFrom(ValueLayout.JAVA_LONG, rngSeed);
			MemorySegment pal = arena.allocate(ValueLayout.JAVA_INT, 256);
			MemorySegment.copy(palette, 0, pal, ValueLayout.JAVA_INT, 0, palette.length);
			MemorySegment plen = arena.allocateFrom(ValueLayout.JAVA_INT, palette.length);
			MemorySegment alpha = arena.allocate(ValueLayout.JAVA_INT);
			int rc;
			try {
				rc = (int) NQuantNative.nq_remap_ragged.invokeExact(NQuantNative.context(device), kind(), in, w, h, 1, nMaxColors, pal, plen, 1,
					dither ? 1 : 0, seed, outs, MemorySegment.NULL, alpha);
			} catch (Throwable t) {
				throw new Exception(t);
			}
			if (rc != 0)
				throw new Exception("nq_remap_ragged failed (" + rc + "): " + NQuantNative.lastError());
			hasAlpha = alpha.get(ValueLayout.JAVA_INT, 0) != 0;
			this.palette = palette.clone();
			return out.toArray(ValueLayout.JAVA_INT);
		}
	}

	/** boolean hasAlpha() (PnnQuantizer.java:458). */
	public boolean hasAlpha() {
		return hasAlpha;
	}

	/** The palette pnnquan produced in the last convert call. */
	public int[] getPalette() {
		return palette.clone();
	}

	/**
	 * The reference converts a set of files by constructing one quantizer per file in a loop (MainActivity.java:190-194).
	 * The GPU wants them together: hundreds of images share one pass over every stage (the merge loop and the dither are
	 * latency bound per image), and with devices.length > 1 the batch is spread over the GPUs of the node through a
	 * dynamic queue (nq_convert_batch_multi; no collective, the images are independent).
	 *
	 * @param lab      false: PnnQuantizer, true: PnnLABQuantizer
	 * @param images   equally sized ARGB images, width*height ints each
	 * @param rngSeeds one seed per image (PnnLABQuantizer), or null
	 * @param devices  CUDA device ordinals to use, e.g. {0} or {0,1,2,3,4,5,6,7}
	 * @param palettesOut optional, images.length entries: receives each image's palette
	 * @return the quantized images, the int[]s the reference hands to Bitmap.createBitmap (PnnQuantizer.java:455)
	 */
	public static int[][] convertBatch(boolean lab, int[][] images, int width, int height, int nMaxColors, boolean dither,
	                                   long[] rngSeeds, int[] devices, int[][] palettesOut) throws Exception {
		final int n = images.length;
		final long npix = (long) width * height;
		try (Arena arena = Arena.ofConfined()) {
			MemorySegment in = arena.allocate(ValueLayout.JAVA_INT, npix * n);
			for (int i = 0; i < n; ++i) {
				if (images[i].length != npix)
					throw new IllegalArgumentException("image " + i + " does not hold width*height pixels");
				MemorySegment.copy(images[i], 0, in, ValueLayout.JAVA_INT, 4L * npix * i, (int) npix);
			}
			MemorySegment out = arena.allocate(ValueLayout.JAVA_INT, npix * n);
			MemorySegment pal = arena.allocate(ValueLayout.JAVA_INT, 256L * n);
			MemorySegment plen = arena.allocate(ValueLayout.JAVA_INT, n);
			MemorySegment seeds = rngSeeds == null ? MemorySegment.NULL : arena.allocateFrom(ValueLayout.JAVA_LONG, rngSeeds);
			MemorySegment ctxs = arena.allocate(ValueLayout.ADDRESS, devices.length);
			for (int g = 0; g < devices.length; ++g)
				ctxs.setAtIndex(ValueLayout.ADDRESS, g, NQuantNative.context(devices[g]));
			int rc;
			try {
				rc = (int) NQuantNative.nq_convert_batch_multi.invokeExact(ctxs, devices.length,
					lab ? NQuantNative.NQ_KIND_PNNLAB : NQuantNative.NQ_KIND_PNN, in, n, width, height, nMaxColors, dither ? 1 : 0,
					seeds, out, pal, plen, MemorySegment.NULL, 0);
			} catch (Throwable t) {
				throw new Exception(t);
			}
			if (rc != 0)
				throw new Exception("nq_convert_batch_multi failed (" + rc + "): " + NQuantNative.lastError());
			int[][] res = new int[n][];
			for (int i = 0; i < n; ++i) {
				res[i] = out.asSlice(4L * npix * i, 4L * npix).toArray(ValueLayout.JAVA_INT);
				if (palettesOut != null)
					palettesOut[i] = pal.asSlice(4L * 256 * i, 4L * plen.getAtIndex(ValueLayout.JAVA_INT, i)).toArray(ValueLayout.JAVA_INT);
			}
			return res;
		}
	}

	/**
	 * The same for images of DIFFERENT sizes (a folder of photos as it comes): image i is widths[i] x heights[i] pixels.
	 * One call over every image (nq_convert_ragged_multi), so images of all sizes share the pipeline instead of one call per
	 * size; each image gets exactly what convert() gives it alone. Sides must be 1..65535. Like the rest of this package,
	 * written against the C ABI and not compiled here (no JDK in the build image).
	 */
	public static int[][] convertBatch(boolean lab, int[][] images, int[] widths, int[] heights, int nMaxColors, boolean dither,
	                                   long[] rngSeeds, int[] devices, int[][] palettesOut) throws Exception {
		final int n = images.length;
		if (widths.length != n || heights.length != n)
			throw new IllegalArgumentException("one width and one height per image");
		try (Arena arena = Arena.ofConfined()) {
			MemorySegment ins = arena.allocate(ValueLayout.ADDRESS, n);
			MemorySegment outs = arena.allocate(ValueLayout.ADDRESS, n);
			MemorySegment[] out = new MemorySegment[n];
			for (int i = 0; i < n; ++i) {
				final long npix = (long) widths[i] * heights[i];
				if (images[i].length != npix)
					throw new IllegalArgumentException("image " + i + " does not hold widths[i]*heights[i] pixels");
				ins.setAtIndex(ValueLayout.ADDRESS, i, arena.allocateFrom(ValueLayout.JAVA_INT, images[i]));
				out[i] = arena.allocate(ValueLayout.JAVA_INT, npix);
				outs.setAtIndex(ValueLayout.ADDRESS, i, out[i]);
			}
			MemorySegment w = arena.allocateFrom(ValueLayout.JAVA_INT, widths);
			MemorySegment h = arena.allocateFrom(ValueLayout.JAVA_INT, heights);
			MemorySegment pal = arena.allocate(ValueLayout.JAVA_INT, 256L * n);
			MemorySegment plen = arena.allocate(ValueLayout.JAVA_INT, n);
			MemorySegment seeds = rngSeeds == null ? MemorySegment.NULL : arena.allocateFrom(ValueLayout.JAVA_LONG, rngSeeds);
			MemorySegment ctxs = arena.allocate(ValueLayout.ADDRESS, devices.length);
			for (int g = 0; g < devices.length; ++g)
				ctxs.setAtIndex(ValueLayout.ADDRESS, g, NQuantNative.context(devices[g]));
			int rc;
			try {
				rc = (int) NQuantNative.nq_convert_ragged_multi.invokeExact(ctxs, devices.length,
					lab ? NQuantNative.NQ_KIND_PNNLAB : NQuantNative.NQ_KIND_PNN, ins, w, h, n, nMaxColors, dither ? 1 : 0,
					seeds, outs, pal, plen, MemorySegment.NULL, 0);
			} catch (Throwable t) {
				throw new Exception(t);
			}
			if (rc != 0)
				throw new Exception("nq_convert_ragged_multi failed (" + rc + "): " + NQuantNative.lastError());
			int[][] res = new int[n][];
			for (int i = 0; i < n; ++i) {
				res[i] = out[i].toArray(ValueLayout.JAVA_INT);
				if (palettesOut != null)
					palettesOut[i] = pal.asSlice(4L * 256 * i, 4L * plen.getAtIndex(ValueLayout.JAVA_INT, i)).toArray(ValueLayout.JAVA_INT);
			}
			return res;
		}
	}

	/** Quantizer objects share their thread's context (NQuantNative.context); nothing to release per object. */
	@Override
	public void close() {
	}

	/** Returns the device memory of this thread's contexts; they are re-created on demand. */
	public static void releaseNativeContexts() {
		NQuantNative.releaseContexts();
	}
}

package com.android.nQuant.b200;

import java.lang.foreign.Arena;
import java.lang.foreign.FunctionDescriptor;
import java.lang.foreign.Linker;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.SymbolLookup;
import java.lang.foreign.ValueLayout;
import java.lang.invoke.MethodHandle;

/**
 * java.lang.foreign (JDK 22+) binding of include/nquant_b200.h -- the C ABI of libnquant_b200.so.
 * No JNI glue is needed: every entry point takes plain pointers and sizes.
 *
 * NOT COMPILED IN THIS REPOSITORY'S BUILD IMAGE (it has no JDK). The same ABI is exercised through
 * ctypes by nquant_android_b200/_lib.py and tests/test_abi.py; the descriptors below mirror that
 * file one to one.
 */
final class NQuantNative {
	static final int NQ_KIND_PNN = 0;      // com.android.nQuant.PnnQuantizer
	static final int NQ_KIND_PNNLAB = 1;   // com.android.nQuant.PnnLABQuantizer

	private static final Linker LINKER = Linker.nativeLinker();
	private static final SymbolLookup LIB = SymbolLookup.libraryLookup(
		System.getProperty("nquant.b200.lib", "libnquant_b200.so"), Arena.global());

	private static MethodHandle h(String name, FunctionDescriptor fd) {
		return LINKER.downcallHandle(LIB.find(name).orElseThrow(() -> new UnsatisfiedLinkError(name)), fd);
	}

	private static final ValueLayout.OfInt I = ValueLayout.JAVA_INT;
	private static final ValueLayout.OfLong L = ValueLayout.JAVA_LONG;
	private static final java.lang.foreign.AddressLayout P = ValueLayout.ADDRESS;

	// nq_ctx* nq_create(int device); void nq_destroy(nq_ctx*); const char* nq_last_error(void)
	static final MethodHandle nq_create = h("nq_create", FunctionDescriptor.of(P, I));
	static final MethodHandle nq_destroy = h("nq_destroy", FunctionDescriptor.ofVoid(P));
	static final MethodHandle nq_last_error = h("nq_last_error", FunctionDescriptor.of(P));
	// int nq_convert(ctx, kind, argb_in, width, height, n_max_colors, dither, rng_seed, argb_out, palette_out, palette_len, has_alpha)
	static final MethodHandle nq_convert = h("nq_convert", FunctionDescriptor.of(I, P, I, P, I, I, I, I, L, P, P, P, P));
	// int nq_convert_batch(ctx, kind, argb_in, n_images, width, height, n_max_colors, dither, rng_seeds, argb_out, palettes_out, palette_lens, has_alpha)
	static final MethodHandle nq_convert_batch = h("nq_convert_batch", FunctionDescriptor.of(I, P, I, P, I, I, I, I, I, P, P, P, P, P));
	// int nq_convert_batch_multi(contexts, n_contexts, kind, argb_in, n_images, width, height, n_max_colors, dither, rng_seeds,
	//                            argb_out, palettes_out, palette_lens, has_alpha, queue_images): one batch over several GPUs
	static final MethodHandle nq_convert_batch_multi = h("nq_convert_batch_multi",
		FunctionDescriptor.of(I, P, I, I, P, I, I, I, I, I, P, P, P, P, P, I));
	// int nq_convert_ragged_multi(contexts, n_contexts, kind, argb_in[], widths, heights, n_images, n_max_colors, dither,
	//                             rng_seeds, argb_out[], palettes_out, palette_lens, has_alpha, queue_images): images of different sizes
	static final MethodHandle nq_convert_ragged_multi = h("nq_convert_ragged_multi",
		FunctionDescriptor.of(I, P, I, I, P, P, P, I, I, I, P, P, P, P, P, I));
	// int nq_convert_ragged_indexed(ctx, kind, argb_in[], widths, heights, n_images, n_max_colors, dither, rng_seeds,
	//                               index_out[], argb_out[] (NULL: colours not returned), palettes_out, palette_lens, has_alpha)
	static final MethodHandle nq_convert_ragged_indexed = h("nq_convert_ragged_indexed",
		FunctionDescriptor.of(I, P, I, P, P, P, I, I, I, P, P, P, P, P, P));
	// int nq_remap_ragged(ctx, kind, argb_in[], widths, heights, n_images, n_max_colors, palettes_in, palette_lens_in, n_palettes,
	//                     dither, rng_seeds, argb_out[] (or NULL), index_out[] (or NULL), has_alpha): dither to the caller's palettes
	static final MethodHandle nq_remap_ragged = h("nq_remap_ragged",
		FunctionDescriptor.of(I, P, I, P, P, P, I, I, P, P, I, I, P, P, P, P));
	// int nq_device_count(void)
	static final MethodHandle nq_device_count = h("nq_device_count", FunctionDescriptor.of(I));
	// int nq_set_spec_dither(ctx, on, segment, warmup): speculative segment-parallel error diffusion, on by default (DESIGN.md 7.1)
	static final MethodHandle nq_set_spec_dither = h("nq_set_spec_dither", FunctionDescriptor.of(I, P, I, I, I));

	/**
	 * One nq_ctx per (thread, GPU), shared by every quantizer object of that thread: a context owns the device workspace
	 * (about 7.5 MB per image in flight plus the 256 MiB RGB->Lab table per device), so it is created once and reused,
	 * not once per image. Contexts are not re-entrant, like the reference's quantizer objects (PnnQuantizer.java:18-33).
	 */
	static final ThreadLocal<java.util.HashMap<Integer, MemorySegment>> CONTEXTS = ThreadLocal.withInitial(java.util.HashMap::new);

	static MemorySegment context(int device) {
		return CONTEXTS.get().computeIfAbsent(device, d -> {
			try {
				MemorySegment c = (MemorySegment) nq_create.invokeExact((int) d);
				if (c.equals(MemorySegment.NULL))
					throw new IllegalStateException("nq_create: " + lastError());
				return c;
			} catch (RuntimeException e) {
				throw e;
			} catch (Throwable t) {
				throw new IllegalStateException(t);
			}
		});
	}

	/** Destroys this thread's contexts (device memory is returned); they are re-created on demand. */
	static void releaseContexts() {
		for (MemorySegment c : CONTEXTS.get().values()) {
			try {
				nq_destroy.invokeExact(c);
			} catch (Throwable ignored) {
			}
		}
		CONTEXTS.get().clear();
	}

	static String lastError() {
		try {
			MemorySegment s = (MemorySegment) nq_last_error.invokeExact();
			return s.reinterpret(4096).getString(0);
		} catch (Throwable t) {
			return t.toString();
		}
	}

	private NQuantNative() {
	}
}

/* nquant_b200.h -- C ABI of the B200 implementation of nQuant's quantizer hot path.
 *
 * The reference (mcychan/nQuant.android) is pure Java and has no FFI today; these are the entry
 * points a JNI / java.lang.foreign binding of its public surface would bind. Each one names the
 * reference interface it stands in for (paths relative to
 * nQuant.master/src/main/java/com/android/nQuant/). INTEGRATION.md shows the Java-side stub.
 *
 * Pixel layout everywhere: row-major, non-premultiplied 0xAARRGGBB, bidx = x + y*width -- the int[]
 * the reference fills with Bitmap.getPixels (PnnQuantizer.java:39-44) and hands to
 * Bitmap.createBitmap (PnnQuantizer.java:455).
 *
 * Ownership: the caller owns every buffer; the library keeps no pointer after a call returns.
 * Threading: one nq_ctx per (thread, GPU). Distinct contexts run concurrently; one context is not
 * re-entrant (the reference's quantizer instances are not thread-safe either, PnnQuantizer.java:18-33).
 * Errors: 0 on success, a negative NQ_ERR_* otherwise; nq_last_error() returns the thread's message.
 * There is no CPU fallback: without a usable CUDA device every call fails with NQ_ERR_CUDA.
 */
#ifndef NQUANT_B200_H
#define NQUANT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NQ_KIND_PNN 0     /* com.android.nQuant.PnnQuantizer    (PnnQuantizer.java:16)    */
#define NQ_KIND_PNNLAB 1  /* com.android.nQuant.PnnLABQuantizer (PnnLABQuantizer.java:17) */

#define NQ_OK 0
#define NQ_ERR_CUDA (-1)         /* CUDA runtime failure, or no device                                  */
#define NQ_ERR_ARG (-2)          /* bad argument (null buffer, size <= 0, nMaxColors < 2 or > 256, ...) */
#define NQ_ERR_COLOR (-3)        /* the reference would throw: ColorUtils.setAlphaComponent rejects an
                                    alpha outside 0..255 (CIELABConvertor.java:79)                        */
#define NQ_ERR_UNSUPPORTED (-4)  /* a branch of the reference this build does not cover yet             */
#define NQ_ERR_NOMEM (-5)

typedef struct nq_ctx nq_ctx;

/* Number of CUDA devices visible to the process (0 when there is none). */
int nq_device_count(void);

/* Create / destroy a context bound to one GPU. Stands in for constructing a quantizer object:
 * `new PnnQuantizer(fname)` (PnnQuantizer.java:35), `new PnnLABQuantizer(fname)`
 * (PnnLABQuantizer.java:24) -- the pixels themselves are passed per call instead of being read from a
 * file/Bitmap (PnnQuantizer.java:39-49). Returns NULL on failure. */
nq_ctx* nq_create(int device);
void nq_destroy(nq_ctx* ctx);

/* Order this context's work with a caller-owned CUDA stream (a cudaStream_t passed as void*): a call starts after
 * everything already enqueued on that stream and the stream continues only after the call's last kernel and copy, so a
 * host framework can feed and time the library with its own kernels and events. NULL is CUDA's legacy default stream
 * (stream handle 0, e.g. torch.cuda.default_stream().cuda_stream). Internally a call fans out over the context's own
 * streams (chunks of the batch: copies, histogram / merge loop and dither overlap). nq_reset_stream goes back to the
 * context's private non-blocking stream (the state after nq_create). */
int nq_set_stream(nq_ctx* ctx, void* cuda_stream);
int nq_reset_stream(nq_ctx* ctx);

/* Images per chunk of a batch call (0 = automatic). A batch is cut into chunks that move through the stages as a
 * pipeline: host->device copy, scan/histogram/find_nn/merge, dither, device->host copy each run on their own stream. */
int nq_set_chunk_images(nq_ctx* ctx, int images);

/* Thread-local message of the last failing call. */
const char* nq_last_error(void);

/* `Bitmap convert(int nMaxColors, boolean dither) throws Exception` (PnnQuantizer.java:409-456,
 * inherited by PnnLABQuantizer) on one image held in HOST memory.
 *   kind          NQ_KIND_PNN or NQ_KIND_PNNLAB
 *   argb_in       width*height source pixels (never modified; the reference edits its private copy)
 *   n_max_colors  2..256
 *   dither        the reference's `dither` flag
 *   rng_seed      seed of the java.util.Random that PnnLABQuantizer.closestColorIndex draws from
 *                 (PnnLABQuantizer.java:22,467 -- unseeded and static in the reference, injected here so
 *                 runs are reproducible); ignored by NQ_KIND_PNN
 *   argb_out      width*height result pixels: palette colours, i.e. the int[] the reference passes to
 *                 Bitmap.createBitmap (PnnQuantizer.java:455)
 *   palette_out   optional, room for 256 entries; the palette `pnnquan` produced
 *   palette_len   optional
 *   has_alpha     optional; `boolean hasAlpha()` (PnnQuantizer.java:458-460) after the call */
int nq_convert(nq_ctx* ctx, int kind, const uint32_t* argb_in, int width, int height, int n_max_colors, int dither,
               uint64_t rng_seed, uint32_t* argb_out, uint32_t* palette_out, int* palette_len, int* has_alpha);

/* The same call over a batch of equally sized images in HOST memory (one quantizer object per
 * image in the reference, MainActivity.java:193-194 in a loop). Image i lives at
 * argb_in + i*width*height; rng_seeds may be NULL (seed 0 for every image). palettes_out (optional)
 * holds 256 entries per image, palette_lens / has_alpha (optional) one int per image. */
int nq_convert_batch(nq_ctx* ctx, int kind, const uint32_t* argb_in, int n_images, int width, int height, int n_max_colors,
                     int dither, const uint64_t* rng_seeds, uint32_t* argb_out, uint32_t* palettes_out, int* palette_lens,
                     int* has_alpha);

/* The same batch over SEVERAL GPUs of one node: contexts[g] was created with nq_create(device g) (or several contexts on one
 * device). The images are independent (every `convert` of the reference is, PnnQuantizer.java:18-33), so there is no
 * collective: one host thread per context pulls pieces of `queue_images` images from a shared queue and converts them
 * with nq_convert_batch; a context that finishes early takes the next piece. queue_images == 0 cuts the batch into one
 * piece per context (best when the images cost about the same: the merge loop and the dither want hundreds of images
 * in flight per GPU); smaller pieces balance batches whose images differ a lot in occupied histogram bins. Results land
 * at the image's own index whichever GPU converted it. Host buffers (pinned memory makes the copies overlap). */
int nq_convert_batch_multi(nq_ctx** contexts, int n_contexts, int kind, const uint32_t* argb_in, int n_images, int width, int height,
                           int n_max_colors, int dither, const uint64_t* rng_seeds, uint32_t* argb_out, uint32_t* palettes_out,
                           int* palette_lens, int* has_alpha, int queue_images);

/* As nq_convert_batch, but argb_in / argb_out are DEVICE pointers on the context's GPU (16-byte
 * aligned). For callers that already hold the pixels in HBM; rng_seeds, palettes_out, palette_lens and
 * has_alpha stay host pointers. Work is enqueued on the context's stream and the call returns after
 * the stream has drained. */
int nq_convert_batch_device(nq_ctx* ctx, int kind, const uint32_t* d_argb_in, int n_images, int width, int height,
                            int n_max_colors, int dither, const uint64_t* rng_seeds, uint32_t* d_argb_out,
                            uint32_t* palettes_out, int* palette_lens, int* has_alpha);

/* A batch of images of DIFFERENT sizes in HOST memory: image i is widths[i] x heights[i] pixels at argb_in[i], its result
 * goes to argb_out[i] (the reference's "one quantizer per file" loop, MainActivity.java:190-194, as one call). kind,
 * n_max_colors and dither apply to every image; rng_seeds, palettes_out (256 entries per image), palette_lens and has_alpha
 * as in nq_convert_batch. Each image gets exactly what nq_convert gives it alone; nq_get_image_info(ctx, i, ..) and the
 * debug getters address image i of the call. Every side must be 1..65535. The images share one pass through the
 * pipeline, so a folder of mixed sizes keeps the GPU as full as a batch of one size does; the workspace is laid out for
 * the largest image of the call (see DESIGN.md section 3). */
int nq_convert_ragged(nq_ctx* ctx, int kind, const uint32_t* const* argb_in, const int* widths, const int* heights,
                      int n_images, int n_max_colors, int dither, const uint64_t* rng_seeds, uint32_t* const* argb_out,
                      uint32_t* palettes_out, int* palette_lens, int* has_alpha);

/* The same with DEVICE buffers on the context's GPU: the images packed back to back (image i starts at pixel
 * sum_{j<i} widths[j]*heights[j]), base pointers 16-byte aligned, e.g. torch.cat of the flattened images. */
int nq_convert_ragged_device(nq_ctx* ctx, int kind, const uint32_t* d_argb_in, const int* widths, const int* heights,
                             int n_images, int n_max_colors, int dither, const uint64_t* rng_seeds, uint32_t* d_argb_out,
                             uint32_t* palettes_out, int* palette_lens, int* has_alpha);

/* nq_convert_ragged over several contexts with the dynamic queue of nq_convert_batch_multi (pieces of queue_images
 * images, 0 = one piece per context). */
int nq_convert_ragged_multi(nq_ctx** contexts, int n_contexts, int kind, const uint32_t* const* argb_in, const int* widths,
                            const int* heights, int n_images, int n_max_colors, int dither, const uint64_t* rng_seeds,
                            uint32_t* const* argb_out, uint32_t* palettes_out, int* palette_lens, int* has_alpha, int queue_images);

/* Stage hook (parity + profiling): GilbertCurve.dither / BlueNoise.dither with a caller-supplied
 * palette (PnnQuantizer.java:393-407, PnnLABQuantizer.java:492-522). Runs the alpha scan and the
 * histogram-derived scalars as convert() would, but replaces the palette pnnquan produced by
 * palette_in before dithering. Host buffers. */
int nq_dither_with_palette(nq_ctx* ctx, int kind, const uint32_t* argb_in, int width, int height, int n_max_colors,
                           int dither, uint64_t rng_seed, const uint32_t* palette_in, int palette_len, uint32_t* argb_out);

/* Stage hook (parity + profiling): the front of pnnquan alone -- alpha scan (PnnQuantizer.java:411-436), the 65 536-bin
 * histogram with compaction, means and getQuanFn (PnnQuantizer.java:137-191, PnnLABQuantizer.java:134-241) and the initial
 * find_nn sweep (PnnQuantizer.java:196-197, PnnLABQuantizer.java:246-247) -- of one image in HOST memory; no merge loop, no
 * dither. n_bins receives the number of occupied bins; bins5 (optional, capacity x 5 doubles: alpha, c1, c2, c3, count),
 * init_err / init_nn (optional, capacity entries) the state at PnnQuantizer.java:192 and each bin's first nearest
 * neighbour. The scalars (weight, ratio, quan_rt, ...) are available through nq_get_image_info(ctx, 0, ..) afterwards. */
int nq_histogram(nq_ctx* ctx, int kind, const uint32_t* argb_in, int width, int height, int n_max_colors, int* n_bins,
                 double* bins5, float* init_err, int* init_nn, int capacity);

/* Generalized Hilbert visiting order for a width x height image (GilbertCurve.java:282-334,
 * 356-365): order_out[n] = x + y*width of the n-th pixel diffusePixel is called on. Host buffer. Computed on the host
 * by the same position -> pixel function (csrc/nq_gilbert.h) that builds the convert calls' tables on the device. */
int nq_gilbert_order(int width, int height, uint32_t* order_out);

/* ---- introspection of the last batch (parity tests, bench counters) --------------------------- */

/* Per-image facts of the last nq_convert* call on this context. */
typedef struct nq_image_info {
  int has_semi_transparency;   /* hasSemiTransparency (PnnQuantizer.java:431)  */
  int transparent_pixel_index; /* m_transparentPixelIndex (PnnQuantizer.java:420) */
  uint32_t transparent_color;  /* m_transparentColor */
  int maxbins, quan_rt, texicab, is_nano;
  double weight, ratio_init, ratio_merge, pr, pg, pb, pa;
  int g_margin, g_thresold, g_dither_max_q, g_dither_max, g_sorted, g_has_alpha, g_use_saliency;
  float g_beta;
  float bn_weight;
  int palette_len;
  unsigned long long merges, rescans, pair_tests, rng_draws, heap_pops;
  int error;
  unsigned long long full_evals; /* CIELAB merge loop: candidates that reached the trigonometric part of find_nn */
  /* CIELAB merge loop: SM cycles per phase (heap/top, first 32, block tests, screen, full+resolve, merge+rebuild),
     blocks that survived their summary test, candidates that survived the screen */
  unsigned long long merge_cycles[6], live_blocks, screened;
  /* FIFO dither kernel: SM cycles of the serial (consumer) warp, of which waiting for the producer warp, and cycles the
     producer warp waited for ring space */
  unsigned long long dither_cycles[3];
  /* CIELAB merge loop: rounds of rescans (stale heap entries rescanned together, see nq_pnn.cuh), and rescans computed
     in a round but not applied because a merge or the next round came first. `rescans` counts the applied ones only. */
  unsigned long long merge_rounds, rescans_discarded;
  /* CTAs of the merge loop kernel of this image's kind (k_merge_lab or k_merge_rgb, one CTA per image) that one SM holds at
     once, as the occupancy calculator reports it for this device */
  int merge_ctas_per_sm;
} nq_image_info;
int nq_get_image_info(nq_ctx* ctx, int image, nq_image_info* out);
/* sizeof(nq_image_info) as the library was built: lets a binding check its own mirror of the struct. */
int nq_sizeof_image_info(void);

/* Speculative segment-parallel error diffusion (csrc/nq_dither_spec.cuh) for PnnLABQuantizer images with more than 64
 * colours, dither on, no transparency: GilbertCurve.dither (GilbertCurve.java:367-373) is cut into `segment`-pixel
 * pieces of the curve that start from an empty error queue `warmup` pixels early and are validated, in curve order,
 * against the exact state of their predecessor (bit-identical results by construction; images it cannot finish go
 * through the serial kernel, which runs next to it for the images that do not qualify). segment == 0 picks the length
 * from the size of the job (8192, shorter for small batches). ON by default (NQ_SPEC_DITHER=0 in the environment at
 * nq_create, or on == 0 here, leaves every image to the serial kernels).
 * nq_get_spec_stats: images completed by this path, validation rounds, and qualifying images it handed back to the
 * serial kernel, since the context was created. */
int nq_set_spec_dither(nq_ctx* ctx, int on, int segment, int warmup);
int nq_get_spec_stats(nq_ctx* ctx, unsigned long long* images, unsigned long long* rounds, unsigned long long* fallbacks);

/* When enabled (flag != 0) the next calls keep, per image, the compacted bins before merging, the
 * initial find_nn results and the merge sequence, retrievable below. Costs memory and a few copies. */
int nq_set_debug(nq_ctx* ctx, int flag);
/* bins5: maxbins x 5 doubles (alpha, c1, c2, c3, cnt) -- mean colour (r,g,b or L,A,B) and the count
 * after getQuanFn, i.e. the state at PnnQuantizer.java:192 / PnnLABQuantizer.java:218. */
int nq_debug_get_bins(nq_ctx* ctx, int image, double* bins5, float* init_err, int* init_nn);
/* pairs: merges x 2 ints (tb, nb) in merge order (PnnQuantizer.java:240-254). */
int nq_debug_get_merges(nq_ctx* ctx, int image, int* pairs);
/* saliency map of the image (PnnLABQuantizer.java:155-156, 499-508), width*height floats. */
int nq_debug_get_saliencies(nq_ctx* ctx, int image, float* out);

/* Kernels launched by this context since creation (bench.py's gpu_launches). */
unsigned long long nq_kernel_launches(nq_ctx* ctx);
/* Device time per stage, measured with CUDA events on the streams the stages run on and accumulated over the
 * chunks and calls since the last reset (chunks overlap: the sum can exceed the wall time of the call). ms[6] / launches[6]: 0 alpha scan, 1 histogram (+compaction), 2 initial
 * find_nn sweep, 3 merge loop, 4 dither setup + saliency, 5 dither (Gilbert pass + blue-noise pass). */
int nq_get_stage_times(nq_ctx* ctx, double* ms, unsigned long long* launches, int reset);
/* Device time of single kernels, each bracketed by its own pair of CUDA events on the stream it is launched on
 * (bench.py's roofline line): ms[4] / launches[4]: 0 k_spec_run (stage 6 of the speculative dither, one entry per launch),
 * 1 k_dither_fifo, 2 k_dither_sorted, 3 k_merge_lab / k_merge_rgb. Accumulated since the last reset. */
int nq_get_kernel_times(nq_ctx* ctx, double* ms, unsigned long long* launches, int reset);
/* Device-side math probe (tests): evaluates the shared nq_math.h kernels ON THE GPU.
 * fn: 0 pow(x,y) 1 exp 2 tanh 3 cbrt 4 atan2(x,y) 5 sin 6 cos. n elements, host buffers. */
int nq_debug_math(nq_ctx* ctx, int fn, const double* x, const double* y, double* out, int n);

/* Device-side CIEDE2000 probe (tests): the L', C', H' and R_T terms of find_nn (PnnLABQuantizer.java:86-104,
 * CIELABConvertor.java:91-194) for n colour pairs, through the SAME routine the merge kernels use (plain-double
 * filter in front of the correctly rounded kernels). lab1/lab2: n x (L, A, B) floats; out: n x 4 floats;
 * n_exact (optional): how many pairs needed the exact path. Host buffers. */
int nq_debug_ciede(nq_ctx* ctx, const float* lab1, const float* lab2, float* out, int* n_exact, int n);

/* Fills a device buffer with the synthetic test image of SURVEY.md 8(d) (see
 * nquant_android_b200/synth.py for the definition) -- used by bench.py so inputs can be created in
 * HBM. cls: 0 smooth, 1 noisy, 2 rand; alpha_mode: 0 opaque, 1 transparent block, 2 semi. */
int nq_synth_device(nq_ctx* ctx, uint32_t* d_out, int n_images, int width, int height, int cls, int alpha_mode,
                    uint64_t seed0);

#ifdef __cplusplus
}
#endif
#endif /* NQUANT_B200_H */

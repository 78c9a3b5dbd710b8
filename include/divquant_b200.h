/* divquant_b200.h -- C ABI of the B200-native DivQuant colour quantizer (libdivquant_b200.so).
 *
 * This is the drop-in boundary for the ONE hot path of caomw/ClusteringSegmentation-1 that this
 * repository accelerates: the DivQuant quantizer (24-bit colour histogram -> divisive variance split
 * with local 2-means -> nearest-palette remap).  Every entry point is plain C: pointers and sizes,
 * no C++ or torch types.  Each one names the reference interface it replaces (file:line under the
 * reference root).  INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Pixel format everywhere: uint32_t 0xAARRGGBB; alpha is ignored on input and zero on output
 * (DivQuantMapColors.cpp:125-127, 523-527).
 *
 * Error behaviour follows the reference: void functions, no error codes; fatal conditions (CUDA
 * failure, out of memory, internal inconsistency) print to stderr and abort()
 * (check_mem, DivQuantMapColors.cpp:43-51; DivQuantCluster.cpp:1021-1026).  There is no CPU
 * fallback: without a usable sm_100a device the library aborts with a message.
 */
#ifndef DIVQUANT_B200_H
#define DIVQUANT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* The library is built with hidden visibility; only what this header (and the reference-named shim)
 * declares is exported. */
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

/* ------------------------------------------------------------------------------------------------
 * 1. Reference-signature entry points (HOST pointers, default context on the current CUDA device).
 *    Same names as the reference with a dq_ prefix; same argument order and meaning.
 * ---------------------------------------------------------------------------------------------- */

/* Replaces  extern "C" quant_recurse        DivQuant/quant_util.h:10, quant_util.cpp:20-158.
 * Quantize to *numClustersPtr colours (max_iters 10, 8 bits, no decimation), drop duplicate palette
 * words (first occurrence wins), remap every pixel.  *numClustersPtr: in = requested K, out = actual.
 * outPixelsPtr and outColortablePtr must hold numPixels and K words. */
void dq_quant_recurse(uint32_t numPixels, const uint32_t *inPixelsPtr, uint32_t *outPixelsPtr,
                      uint32_t *numClustersPtr, uint32_t *outColortablePtr, int allPixelsUnique);

/* Replaces  quant_varpart_fast              DivQuant/DivQuantHeader.h:82-94, DivQuantCluster.cpp:1099-1179.
 * tmpPixels (capacity numPixels) is scratch exactly as in the reference and is left unspecified. */
void dq_quant_varpart_fast(uint32_t numPixels, const uint32_t *inPixels, uint32_t *tmpPixels, uint32_t numRows,
                           uint32_t numCols, uint32_t *numClustersPtr, uint32_t *colortablePtr, int num_bits,
                           int dec_factor, int max_iters, int allPixelsUnique);

/* Replaces  map_colors_mps                  DivQuant/DivQuantHeader.h:61, DivQuantMapColors.cpp:243-539.
 * The colortable is read, never written. */
void dq_map_colors_mps(const uint32_t *inPixelsPtr, uint32_t numPixels, uint32_t *outPixelsPtr,
                       const uint32_t *colortablePtr, int colormapSize);

/* Replaces  calc_color_table                DivQuant/DivQuantHeader.h:63-70, DivQuantMapColors.cpp:82-203.
 * The reference returns `new double[U]`; a C ABI cannot, so the caller passes weightsOut (capacity:
 * the number of sampled pixels, ceil(numRows/dec)*ceil(numCols/dec)).  Unique colours are emitted in the
 * reference's order (hash bucket ascending, most recently first-seen colour first inside a bucket).
 * Returns 0, or -1 when dec_factor <= 0 (the reference prints a message and returns NULL). */
int dq_calc_color_table(const uint32_t *inPixels, uint32_t numPixels, uint32_t *outPixels, uint32_t numRows,
                        uint32_t numCols, int dec_factor, int *num_colors, double *weightsOut);

/* Replaces  cut_bits                        DivQuant/DivQuantHeader.h:72-79, DivQuantUni.cpp:28-100.
 * In-place (inPixels == outPixels) is allowed.  Invalid bit counts: message on stderr, no output. */
void dq_cut_bits(const uint32_t *inPixels, uint32_t numPixels, uint32_t *outPixels, unsigned char num_bits_red,
                 unsigned char num_bits_green, unsigned char num_bits_blue);

/* Replaces  get_double_scale                DivQuant/DivQuantHeader.h:55-57, DivQuantMapColors.cpp:205-220. */
double dq_get_double_scale(const uint32_t *inPixels, uint32_t numPixels);

/* Replaces  validate_num_bits               DivQuant/DivQuantHeader.h:96, DivQuantMisc.cpp:36-46. */
int dq_validate_num_bits(unsigned char num_bits);

/* When non-zero (default 1) dq_quant_recurse prints the reference's two timing lines on stdout
 * (quant_util.cpp:62-66, 141-145).  Also settable with DIVQUANT_B200_TIMINGS=0 in the environment. */
void dq_set_display_timings(int enabled);

/* ------------------------------------------------------------------------------------------------
 * 2. Explicit contexts and DEVICE-pointer entry points (what a pipeline that already keeps frames in
 *    HBM, and bench.py's device-resident leg, call).  One context = one CUDA device + one stream +
 *    its scratch (the 64 MB direct colour table, point buffers, controller state).  A context is not
 *    thread-safe; use one per thread/stream.
 * ---------------------------------------------------------------------------------------------- */
typedef struct dq_context dq_context;

/* device < 0 : use the current device. Aborts on failure like every other entry point. */
dq_context *dq_context_create(int device);
void dq_context_destroy(dq_context *ctx);
/* The lazily created context behind the section-1 entry points. */
dq_context *dq_default_context(void);
/* cudaStream_t of the context, as a void* (so that this header needs no CUDA headers). */
void *dq_context_stream(dq_context *ctx);
void dq_context_synchronize(dq_context *ctx);

/* What the last call on a context did (for tests, bench.py and tracing). */
typedef struct {
  uint32_t num_pixels;
  uint32_t num_points;       /* U: unique colours (or pixels on the allPixelsUnique path)   */
  uint32_t requested_colors; /* K asked for                                                */
  uint32_t actual_colors;    /* palette entries returned                                   */
  uint32_t empty_clusters;   /* clusters dropped as empty (DivQuantCluster.cpp:1058-1069)  */
  uint32_t split_rounds;     /* rounds of the persistent split kernel                      */
  uint32_t splits_computed;  /* splits evaluated, speculative ones included                */
  uint32_t remap_path;       /* 0 none, 1 brute force over pixels, 2 unique-colour table   */
  uint32_t kernel_launches;  /* kernels launched by the call                               */
  /* Device time of each stage in milliseconds (CUDA events on the context's stream); only filled
   * while profiling is enabled with dq_context_set_profiling, else 0:
   * [0] hist_insert  [1] hist_collect / points_from_pixels  [2] split kernel
   * [3] map_unique or brute-force map  [4] map_gather  [5] table_clear  [6] whole call */
  float stage_ms[7];
  /* Tie audit of the exact-integer split (inputs above the ordered path's limit): bit d-1 set = a decision of kind d
   * sat inside the rounding noise of the reference's sequential sums (1 axis :388-403, 2 cut :473, 4 hyperplane :683,
   * 8 TSE arg-max :876-887, 16 palette rounding :1050-1052, 32 degenerate TSE order; 64 = NOT audited: more
   * than 512 colours requested on more than 262144 distinct colours, where neither the audited kernel nor the ordered
   * path applies -- requests above 512 colours otherwise always take the ordered path).  0 = the result is the
   * reference's bit for bit.  ordered_rerun = 1: the frame was flagged and computed again in the reference's
   * summation order (so the result is the reference's as well). */
  uint32_t tie_flags;
  uint32_t ordered_rerun;
  /* > 0: only palette roundings (bit 16) and / or cuts (bit 2) were flagged and that many of them were settled by the
   * resolver (csrc/dq_resolve.cu), which recomputes the one node mean each of them hangs on in the reference's own
   * arithmetic: a rounding is rewritten, a cut is confirmed to separate the same points as the reference's.  The result is
   * the reference's, without a re-run.  (A cut that does NOT separate the same points sends the frame to the re-run.) */
  uint32_t tie_resolved;
  /* > 0: that many nodes were cut where the resolver found the reference cuts them (a mean on an integer that the
   * reference's rounding noise puts on the other side), by running the exact-integer split again with those cuts forced. */
  uint32_t cut_overrides;
} dq_call_stats;
void dq_context_last_stats(const dq_context *ctx, dq_call_stats *out);
/* Per-stage CUDA-event timing of dq_quant_recurse_device / _ctx calls (off by default). */
void dq_context_set_profiling(dq_context *ctx, int enabled);
/* Number of CTAs (one per SM) the persistent split kernel of this context occupies; default = all SMs
 * (lowest latency of one call).  Several contexts with num_ctas = SMs / contexts run their latency-bound split
 * phases side by side on one GPU (frame pipeline with lanes, section 2b).  Results do not depend on it.
 * Out-of-range values restore the default.  Environment: DIVQUANT_B200_SPLIT_CTAS. */
void dq_context_set_split_ctas(dq_context *ctx, int num_ctas);
/* Weighted inputs (allPixelsUnique = 0) of at most `max_points` unique colours (and K <= 4096) are split by code that
 * adds in the reference's own order (calc_color_table emission order, one sequential double sum per accumulator), so
 * that even decisions that sit exactly on a tie come out as in the reference: bit-exact palettes.  Larger inputs use
 * exact integer sums with the tie audit below, which sends the frames that need it back to the ordered path (it takes up
 * to 262144 colours) -- so the palette is the reference's either way and this limit is a performance knob: the ordered
 * path costs ~0.2 ms for 100 colours, ~1.2 ms for 4096, ~3 ms for 16384, 20 ms for 40 000 (K = 256, sequential chains),
 * the audited integer kernels 0.3-0.5 ms whatever the size.
 * max_points: 0..262144, default 4096 (environment DIVQUANT_B200_EXACT_MAX); dq_context_set_exact_small(ctx, 0)
 * (environment DIVQUANT_B200_EXACT_SMALL=0) turns the ordered path off altogether (flagged frames are then only reported). */
void dq_context_set_exact_max_points(dq_context *ctx, uint32_t max_points);
void dq_context_set_exact_small(dq_context *ctx, int enabled);
/* Inputs above that limit run on exact integer sums, which equal the reference's sequential double sums up to the
 * reference's own rounding noise.  The split kernel audits every decision it takes (axis, cut, hyperplane, TSE
 * arg-max, palette rounding) against first-order bounds of that noise (csrc/dq_tie.cuh).  policy 2 (default): a frame
 * with a decision inside its bound is settled by the resolver (flagged roundings and cuts: any number of colours) or
 * computed again on the ordered path (anything else: up to 262144 colours), so the palette is the reference's either way; 1: only report (dq_call_stats::tie_flags); 0: no audit.  Environment: DIVQUANT_B200_TIE. */
void dq_context_set_tie_policy(dq_context *ctx, int policy);

/* quant_recurse with pixels already resident in HBM.  d_in / d_out are device pointers on the
 * context's device; colortable and numClustersPtr are host pointers.  Synchronous with respect to
 * the host on return (the palette has to come back for the reference's std::sort of it). */
void dq_quant_recurse_device(dq_context *ctx, uint32_t numPixels, const uint32_t *d_in, uint32_t *d_out,
                             uint32_t *numClustersPtr, uint32_t *outColortablePtr, int allPixelsUnique);

/* map_colors_mps with pixels resident in HBM (colortable on the host). Asynchronous on the context's
 * stream except for the small palette upload. prefer_table: 1 = histogram + per-unique-colour table
 * when profitable, 0 = always brute force over pixels. */
void dq_map_colors_device(dq_context *ctx, const uint32_t *d_in, uint32_t numPixels, uint32_t *d_out,
                          const uint32_t *colortablePtr, int colormapSize, int prefer_table);

/* quant_varpart_fast with pixels resident in HBM; palette returned to host memory. */
void dq_quant_varpart_device(dq_context *ctx, uint32_t numPixels, const uint32_t *d_in, uint32_t numRows,
                             uint32_t numCols, uint32_t *numClustersPtr, uint32_t *colortablePtr, int num_bits,
                             int dec_factor, int max_iters, int allPixelsUnique);

/* Host-pointer quant_recurse on an explicit context (what dq_quant_recurse forwards to). */
void dq_quant_recurse_ctx(dq_context *ctx, uint32_t numPixels, const uint32_t *inPixelsPtr, uint32_t *outPixelsPtr,
                          uint32_t *numClustersPtr, uint32_t *outColortablePtr, int allPixelsUnique);

/* Block majority vote (SURVEY.md 8f row 1).  Replaces the numeric part of  genHistogramsForBlocks
 * ClusteringSegmentation/ClusteringSegmentation.cpp:417-563: every superpixelDim x superpixelDim block (clipped at
 * the border; ceil(width/dim) x ceil(height/dim) blocks, ClusteringSegmentationMain.cpp:139-149) is represented
 * by its most frequent quantized pixel.  Ties go to the first maximum in the iteration order of the
 * std::unordered_map<uint32_t,uint32_t> the reference counts in (libstdc++ bucket rule, reproduced on the device).
 * superpixelDim in 1..8.  Host pointers; blocksOut has ceil(width/dim)*ceil(height/dim) words, row-major. */
void dq_block_vote(const uint32_t *quantPixels, uint32_t width, uint32_t height, uint32_t superpixelDim, uint32_t *blocksOut);
void dq_block_vote_device(dq_context *ctx, const uint32_t *d_quantPixels, uint32_t width, uint32_t height,
                          uint32_t superpixelDim, uint32_t *d_blocksOut);
/* The whole numeric front half of genHistogramsForBlocks in one call (ClusteringSegmentation.cpp:397-563): remap the
 * image to `colortable` and vote per block; the quantized image never leaves the GPU unless quantOut != NULL. */
void dq_quant_blocks(const uint32_t *inPixels, uint32_t width, uint32_t height, uint32_t superpixelDim,
                     const uint32_t *colortable, int colormapSize, uint32_t *quantOut, uint32_t *blocksOut);

/* Per-image pixel histogram (SURVEY.md 8f row 2).  Replaces  generatePixelHistogram  superpixels/OpenCVUtil.cpp:736-781
 * (3-channel form: pixel &= 0x00FFFFFF): the (pixel, count) pairs the reference leaves in its unordered_map, here as
 * two arrays sorted by ascending pixel value (a map has no order to mirror).  Returns the number of distinct
 * pixels U; writes min(U, capacity) pairs.  Host pointers. */
uint32_t dq_pixel_histogram(const uint32_t *pixels, uint32_t numPixels, uint32_t *pixelsOut, uint32_t *countsOut, uint32_t capacity);

/* SRM front half (SURVEY.md 8f row 4).  Replaces the edge generation and bucket sort inside  segmentation()
 * SRM/srm.c:135-177, :226-246 : the C4 edge list of an interleaved 8-bit image (colour bytes 0..2 of every pixel,
 * `channels` bytes per pixel, `widthStep` bytes per row) in the reference's generation order, stably sorted by
 * diff = the largest per-channel absolute difference (srm.c:103-121) -- i.e. exactly srm->ordered_pairs, the merge
 * order of the union-find loop that stays on the host (srm.c:181-190).  dq_srm_pair is field-compatible with the
 * reference's `struct my_pair` (SRM/srm.h:5-9).  orderedPairs holds dq_srm_num_pairs(width, height) entries. */
typedef struct {
  uint32_t r1, r2, diff;
} dq_srm_pair;
uint32_t dq_srm_num_pairs(uint32_t width, uint32_t height); /* 2(w-1)(h-1) + (h-1) + (w-1), srm.c:58 */
void dq_srm_sorted_edges(const uint8_t *in, uint32_t width, uint32_t height, uint32_t channels, uint32_t widthStep,
                         dq_srm_pair *orderedPairs);                                       /* host pointers   */
void dq_srm_sorted_edges_device(dq_context *ctx, const uint8_t *d_in, uint32_t width, uint32_t height, uint32_t channels,
                                uint32_t widthStep, dq_srm_pair *d_orderedPairs);          /* device pointers */

/* Label image (SURVEY.md 8f row 2).  Replaces  mapQuantPixelsToColortableIndexes   superpixels/OpenCVUtil.cpp:787-849:
 * every (already quantized) pixel -> index of its colour in the CALLER's palette order, the last duplicate
 * winning; asGreyscale != 0 writes (i<<16 | i<<8 | i) like the reference (indexes must then be < 256).
 * A pixel that is not in the palette is fatal (message + abort; assert(0) in the reference).  Host pointers. */
void dq_colortable_indexes(const uint32_t *quantPixels, uint32_t numPixels, const uint32_t *colortable, int colormapSize,
                           uint32_t *labelsOut, int asGreyscale);
/* Same with device pixel / label buffers on an explicit context. */
void dq_colortable_indexes_device(dq_context *ctx, const uint32_t *d_quantPixels, uint32_t numPixels,
                                  const uint32_t *colortable, int colormapSize, uint32_t *d_labelsOut, int asGreyscale);

/* ------------------------------------------------------------------------------------------------
 * 2a. Pixel-row sharding of ONE image over several GPUs (BASELINE.json config 3; one process per GPU).
 *     Counts are additive over shards and every sum of the divisive phase is an exact integer, so the
 *     palette is independent of the number of shards.  The one exchange runs inside the library (NCCL over NVLink, looked
 *     up with dlopen("libnccl.so.2") at run time, so the copy the process already has -- e.g. PyTorch's -- is used and the
 *     library has no link-time dependency on it).
 * ---------------------------------------------------------------------------------------------- */
/*   rank 0:      dq_rows_unique_id(id)            -> hand the 128 bytes to every rank (any side channel)
 *   every rank:  rows = dq_rows_create(ctx, world, rank, id, list_capacity)          (collective: ncclCommInitRank)
 *   per image:   dq_rows_quant_recurse(rows, d_shard, n_shard, N_total, d_out_shard, &K, palette)
 * One grouped ncclAllGather per image on the context's stream of three fixed-capacity slices per rank: colours, counts
 * and the shard-local first-seen index of every colour (plus the shard's pixel count, from which every rank derives the
 * offset of each shard's rows in the image: rows are contiguous and in rank order).  Unused entries carry count 0: no
 * sizes travel first, no host synchronisation before the palette.  list_capacity >= the largest number of unique colours
 * in any shard (a shard that exceeds it is fatal: message + abort); world x (list_capacity + 1) < 2^32.  world = 1 needs no
 * id and no NCCL.
 * Every rank merges the lists into its direct table, and the minimum over shards of (offset + local first-seen index) into
 * the whole image's first-seen index of every colour; the split runs replicated with the tie audit, and a flagged palette
 * rounding or cut is settled by the resolver (and a forced-cut re-split, which merges the gathered lists again) exactly as
 * in the single-GPU call.  Every rank takes identical decisions from identical data, so the palette stays replicated.
 * Result: the palette and this rank's rows of dq_quant_recurse of the whole image, PROVIDED the single-GPU call takes the
 * exact-integer kernels for it (more unique colours than dq_context_set_exact_max_points, default 4096: every BASELINE
 * configuration) and the frame needs no ordered re-run.  The ordered path (small inputs, and flagged axis / hyperplane /
 * TSE decisions, none of them among the golden frames) needs the whole image in order, which no rank has: such frames stay
 * on exact integer sums and are reported in dq_call_stats::tie_flags with ordered_rerun = 0. */
typedef struct dq_rows dq_rows;
void dq_rows_unique_id(void *out128);
dq_rows *dq_rows_create(dq_context *ctx, int world, int rank, const void *unique_id128, uint32_t list_capacity);
void dq_rows_destroy(dq_rows *rows);
void dq_rows_quant_recurse(dq_rows *rows, const uint32_t *d_shard, uint32_t n_shard, uint64_t total_pixels, uint32_t *d_out_shard,
                           uint32_t *numClustersPtr, uint32_t *outColortablePtr);

/* ------------------------------------------------------------------------------------------------
 * 2b. Frame pipeline: quant_recurse over a stream of frames (BASELINE.json config 4, "batch of frames", and both
 *     legs of bench.py).  Frames are independent units and one frame's critical path (the chain of dependent
 *     passes of the split) leaves most of the GPU idle, so the pipeline runs `lanes` frames side by side: every
 *     lane owns a context and a pair of frame buffers, and one host thread walks each lane's frames, one at a time,
 *     through H2D -> kernels -> D2H.  The split kernels of different lanes occupy disjoint groups of SMs,
 *     histogram / remap kernels and both copy engines fill in around them.  Results are exactly those of dq_quant_recurse frame by
 *     frame (they do not depend on the lane or on split_ctas).
 *     Host buffers should be pinned (cudaHostAlloc / torch pin_memory) for the copies to be asynchronous;
 *     pageable buffers work but serialise.  All pointers of a frame (pixels, numClustersPtr, colortable) must stay
 *     valid until dq_pipeline_wait(ticket) or dq_pipeline_flush() returns.  submit / wait / flush may be called
 *     from one thread at a time.
 * ---------------------------------------------------------------------------------------------- */
typedef struct dq_pipeline dq_pipeline;
/* lanes = frames in flight (1..16); max_pixels = largest HOST frame that will be submitted (0 if only device frames
 * are used); split_ctas = CTAs of each lane's split kernel, 0 = (3/4 of the SMs) / lanes, which leaves the histogram /
 * remap kernels of the other lanes SMs of their own. */
dq_pipeline *dq_pipeline_create_lanes(int device, uint32_t max_pixels, int lanes, int split_ctas);
/* Same with lanes = depth (2..8) and the default SM partition. */
dq_pipeline *dq_pipeline_create(int device, uint32_t max_pixels, int depth);
void dq_pipeline_destroy(dq_pipeline *pipe);
/* Queue one frame with HOST pointers; returns its ticket (0, 1, 2, ... in submission order). */
uint64_t dq_pipeline_submit(dq_pipeline *pipe, uint32_t numPixels, const uint32_t *inPixelsPtr, uint32_t *outPixelsPtr,
                            uint32_t *numClustersPtr, uint32_t *outColortablePtr, int allPixelsUnique);
/* Queue one frame whose pixels are DEVICE pointers on the pipeline's device (no copies; numClustersPtr and
 * outColortablePtr stay host pointers).  d_in must be complete when this is called: lanes run on their own streams. */
uint64_t dq_pipeline_submit_device(dq_pipeline *pipe, uint32_t numPixels, const uint32_t *d_in, uint32_t *d_out,
                                   uint32_t *numClustersPtr, uint32_t *outColortablePtr, int allPixelsUnique);
/* Returns when that frame's outPixels / colortable / numClusters are complete. */
void dq_pipeline_wait(dq_pipeline *pipe, uint64_t ticket);
/* Returns when every submitted frame is complete. */
void dq_pipeline_flush(dq_pipeline *pipe);
/* Device time (CUDA events on the lanes' streams) from the first operation of the first frame to the last
 * operation of the last frame submitted between the previous two flushes, in milliseconds. */
float dq_pipeline_last_elapsed_ms(const dq_pipeline *pipe);
/* Lane 0's context (for dq_context_last_stats). */
dq_context *dq_pipeline_context(dq_pipeline *pipe);
/* Kernels launched since creation (sum over frames and lanes). */
uint64_t dq_pipeline_kernel_launches(const dq_pipeline *pipe);
/* Frames (since creation) whose tie audit raised a flag (dq_call_stats::tie_flags != 0). */
uint64_t dq_pipeline_flagged_frames(const dq_pipeline *pipe);
/* Frames (since creation) that the resolver settled (dq_call_stats::tie_resolved or cut_overrides > 0), and frames that were
 * computed again on the ordered path (dq_call_stats::ordered_rerun = 1). */
uint64_t dq_pipeline_resolved_frames(const dq_pipeline *pipe);
uint64_t dq_pipeline_rerun_frames(const dq_pipeline *pipe);
int dq_pipeline_lanes(const dq_pipeline *pipe);
/* The pipeline's one host thread polls its lanes while they wait for the GPU.  It spins (lowest latency; default) or,
 * with enabled = 1, sleeps 20 us between polling rounds: use it when host cores are scarce (several ranks on one host). */
void dq_pipeline_set_blocking_wait(dq_pipeline *pipe, int enabled);

/* ------------------------------------------------------------------------------------------------
 * 2c. Many small inputs in one call: quant_recurse over num_items independent pixel sets (regions of a segmentation,
 *     tiles of an image, thumbnails) packed end to end.  Item i is pixels [offsets[i], offsets[i+1]) of the input.
 *     Each item's result equals dq_quant_recurse_device on this context for that item alone, bit for bit: its palette
 *     (colortables), its actual K (numClusters) and its remapped pixels, and the same "# empty clusters: n" line on stderr.
 *     An item that the single call would split on the ordered path in shared memory (allPixelsUnique = 0, K <= 512 and at
 *     most min(dq_context_set_exact_max_points, 4096) distinct colours with the ordered path on) is computed by batch
 *     kernels, one CTA per item, in launches whose number does not depend on the number of items; every other item goes
 *     through the single call inside the same call, in item order.
 *   offsets:     HOST array of num_items + 1 non-decreasing words, offsets[num_items] <= numPixels.
 *   numClusters: HOST, num_items words: in = requested K of item i, out = actual.
 *   colortables: HOST, sum of the requested K words; item i's palette starts at the sum of the requested K of items < i.
 * Decreasing offsets, offsets beyond numPixels, an item with no pixels or K = 0 are fatal (message + abort).
 * num_items = 0 does nothing.  Neither form prints timing lines.  Synchronous on return.  Afterwards dq_call_stats is
 * zeroed apart from kernel_launches (all the call launched); dq_context_last_batch_stats tells which path the items took.
 * ---------------------------------------------------------------------------------------------- */
void dq_quant_recurse_batch_device(dq_context *ctx, uint32_t num_items, const uint32_t *offsets, uint32_t numPixels, const uint32_t *d_in,
                                   uint32_t *d_out, uint32_t *numClusters, uint32_t *colortables, int allPixelsUnique);
void dq_quant_recurse_batch_ctx(dq_context *ctx, uint32_t num_items, const uint32_t *offsets, uint32_t numPixels, const uint32_t *inPixels,
                                uint32_t *outPixels, uint32_t *numClusters, uint32_t *colortables, int allPixelsUnique);
typedef struct {
  uint32_t items;              /* num_items of the last batch call                                    */
  uint32_t batched_items;      /* items computed by the batch kernels                                  */
  uint32_t single_call_items;  /* items that went through the single call                              */
  uint32_t empty_clusters;     /* sum over all items                                                   */
  uint32_t kernel_launches;    /* kernels launched by the whole call, single calls included            */
  float host_palette_ms;       /* wall clock of the host's palette handling of the batched items      */
} dq_batch_stats;
void dq_context_last_batch_stats(const dq_context *ctx, dq_batch_stats *out);

/* map_colors_mps over num_items independent pixel sets, each mapped to its OWN palette (the per-region remaps of
 * ClusteringSegmentation.cpp:2434, :3816), optionally with the label image mapQuantPixelsToColortableIndexes makes of the
 * result (OpenCVUtil.cpp:787-849).  Item i is pixels [offsets[i], offsets[i+1]) of the input; its palette is
 * colortables[P_i, P_i + colormapSizes[i]), P_i = the sum of colormapSizes of the items before i (the packing of the
 * quant_recurse batch).  Palettes may hold duplicates, alpha bits, equal r+g+b sums and colours absent from the item.
 *   out:    for every item, bit for bit what dq_map_colors_device (prefer_table = 1) on this context returns for it alone:
 *           alpha ignored on input, zero on output.
 *   labels: NULL = none; else labels[p] = dq_colortable_indexes(out of that item, its palette, asGreyscale = 0)[p]: the
 *           0-based index within the item's palette of the LAST entry whose 24-bit colour equals out[p].
 *   offsets, colormapSizes, colortables: HOST arrays (num_items + 1, num_items and sum of colormapSizes words).
 * An item whose palette has at most 512 entries is mapped by one batch remap launch over 1024-pixel tiles of all such
 * items (an all-batched call is one kernel launch, with or without labels); every other item runs dq_map_colors_device
 * (and, for labels, dq_colortable_indexes_device) in item order inside the same call.
 * Decreasing offsets, offsets beyond numPixels, colormapSizes[i] <= 0 and, with labels, colormapSizes[i] > 24000 are
 * fatal (message + abort) before any device work.  An item with no pixels writes nothing; num_items = 0 does nothing.
 * d_out and d_labels must not overlap d_in or each other.  The _ctx form copies only pixels offsets[0] .. offsets[num_items]
 * and copies labels back only when asked for.  Synchronous on return, no timing lines.  Afterwards dq_call_stats is zeroed
 * apart from kernel_launches; dq_context_last_batch_stats gives items, batched_items (palettes <= 512 entries),
 * single_call_items, empty_clusters = 0, kernel_launches and host_palette_ms (building the search and label tables). */
void dq_map_colors_batch_device(dq_context *ctx, uint32_t num_items, const uint32_t *offsets, uint32_t numPixels,
                                const uint32_t *d_in, uint32_t *d_out, const int *colormapSizes,
                                const uint32_t *colortables, uint32_t *d_labels);
void dq_map_colors_batch_ctx(dq_context *ctx, uint32_t num_items, const uint32_t *offsets, uint32_t numPixels,
                             const uint32_t *inPixels, uint32_t *outPixels, const int *colormapSizes,
                             const uint32_t *colortables, uint32_t *labels);

/* quant_recurse of every region of a tag image, each region to its own palette (the per-region quant_recurse calls of
 * ClusteringSegmentation.cpp:758, :1803, :2789, :3152), optionally with the label image of the result.
 * Region r = the pixels p with tags[p] == r, in index (raster) order; tags[p] >= num_regions = in no region.  With
 * item_r = in at region r's pixels, every region with pixels gets exactly what dq_quant_recurse_batch_device on this
 * context returns for the items item_r in region order with the same K (allPixelsUnique = 0): its palette, its actual K,
 * out at its pixels and the same "# empty clusters: n" lines in the same order.
 *   ks:          HOST, num_regions words, in = requested K (>= 1 for every region), out = actual K (0 for a region with no
 *                pixels, which prints nothing and leaves its palette slot untouched).
 *   colortables: HOST, sum(ks) words; region r's palette starts at the sum of the requested K of regions < r (the batch
 *                packing).
 *   out / labels: written at region pixels only; pixels in no region keep what the buffer held.  labels may be NULL; else
 *                labels[p] = the index of out[p] within its region's returned palette (= dq_colortable_indexes of the
 *                region's output, asGreyscale = 0).
 * The device partitions the pixels by tag (a stable radix sort, one pass per byte: up to 256, 65 536, 2^24 regions), then
 * the regions with pixels go through the quant_recurse batch, and the results are scattered back.  num_regions > 2^24 and
 * ks[r] == 0 for any r are fatal (message + abort) before any device work; num_regions = 0 does nothing.  d_out and
 * d_labels must not overlap d_in, d_tags or each other.  The _ctx form copies pixels, tags, out (and labels when asked)
 * up and out (and labels) down.  Synchronous on return, no timing lines.  Afterwards dq_call_stats is zeroed apart from
 * kernel_launches; dq_context_last_batch_stats gives items = num_regions, batched_items and single_call_items of the
 * regions with pixels, empty_clusters, kernel_launches (all the call launched, sort and scatter included) and
 * host_palette_ms. */
void dq_quant_regions_device(dq_context *ctx, uint32_t numPixels, const uint32_t *d_in, const uint32_t *d_tags,
                             uint32_t num_regions, uint32_t *d_out, uint32_t *ks, uint32_t *colortables, uint32_t *d_labels);
void dq_quant_regions_ctx(dq_context *ctx, uint32_t numPixels, const uint32_t *inPixels, const uint32_t *tags,
                          uint32_t num_regions, uint32_t *outPixels, uint32_t *ks, uint32_t *colortables, uint32_t *labels);

/* map_colors_mps of every region of a tag image, each region to its own palette (the per-region remaps of
 * ClusteringSegmentation.cpp:2434, :3816), optionally with the label image of the result (OpenCVUtil.cpp:787-849): the
 * step after dq_quant_regions once the caller has edited the palettes.
 * Region r = the pixels p with tags[p] == r, in index (raster) order; tags[p] >= num_regions = in no region.  Region r's
 * palette is colortables[P_r, P_r + colormapSizes[r]), P_r = the sum of colormapSizes of the regions before r (the map
 * batch's packing).  Palettes may hold duplicates, alpha bits, equal r+g+b sums and colours absent from the region.
 *   colormapSizes, colortables: HOST arrays (num_regions and sum of colormapSizes words).  colormapSizes[r] == 0 = region
 *                r is not mapped: its pixels are treated like pixels in no region (so dq_quant_regions' returned K, 0 for
 *                a region without pixels, can be passed unchanged).
 *   out:         at every pixel of region r, bit for bit what dq_map_colors_batch_device on this context returns for the
 *                item "pixels of region r" (= map_colors_mps of them against that palette): alpha ignored on input, zero
 *                on output.
 *   labels:      NULL = none; else labels[p] = what the map batch writes for p: the 0-based index within region r's
 *                palette of the LAST entry whose 24-bit colour equals out[p].
 *   Pixels in no region and pixels of unmapped regions keep what out / labels held.
 * The device partitions the pixels of the mapped regions by tag (the sort of dq_quant_regions; the first pass drops the
 * unmapped regions' pixels), the regions with pixels go through the map batch as its items in region order, and the
 * results are scattered back.  A call whose mapped regions all have at most 512 entries launches 3 x passes + 3 kernels
 * (passes = 1 up to 256 regions, 2 up to 65 536, 3 above), whatever the number of regions, with or without labels.
 * num_regions > 2^24, colormapSizes[r] < 0 and, with labels, colormapSizes[r] > 24000 are fatal (message + abort) before
 * any device work; num_regions = 0 or numPixels = 0 does nothing.  d_out and d_labels must not overlap d_in, d_tags or
 * each other.  The _ctx form copies pixels, tags, out (and labels when asked) up and out (and labels) down.  Synchronous
 * on return, no timing lines.  Afterwards dq_call_stats is zeroed apart from kernel_launches; dq_context_last_batch_stats
 * gives items = num_regions, batched_items (palettes <= 512 entries) and single_call_items of the mapped regions with
 * pixels, empty_clusters = 0, kernel_launches (all the call launched, sort and scatter included) and host_palette_ms. */
void dq_map_regions_device(dq_context *ctx, uint32_t numPixels, const uint32_t *d_in, const uint32_t *d_tags,
                           uint32_t num_regions, const int *colormapSizes, const uint32_t *colortables,
                           uint32_t *d_out, uint32_t *d_labels);
void dq_map_regions_ctx(dq_context *ctx, uint32_t numPixels, const uint32_t *inPixels, const uint32_t *tags,
                        uint32_t num_regions, const int *colormapSizes, const uint32_t *colortables,
                        uint32_t *outPixels, uint32_t *labels);

/* ------------------------------------------------------------------------------------------------
 * 3. Test hooks (used by tests/ to compare intermediate results with the oracle).
 * ---------------------------------------------------------------------------------------------- */

/* Field-for-field mirror of oracle_split_record (oracle/divquant_oracle.h). */
typedef struct {
  int32_t new_index, old_index, cut_axis, num_points, new_size, is_last;
  double cut_pos;
  double total_weight, new_weight, old_weight;
  double new_mean[3], old_mean[3];
  double new_var[3], old_var[3];
  double new_tse, old_tse;
} dq_split_record;

/* Runs only the divisive phase on caller-supplied (colour, count) points (host arrays).
 * norm = 1/#sampled pixels.  records (capacity K-1), cluster_mean (K*3) and cluster_size (K) may be NULL.
 * Returns the number of palette entries written to colortable (capacity K). */
uint32_t dq_debug_split_points(dq_context *ctx, const uint32_t *colours, const uint32_t *counts, uint32_t num_points,
                               double norm, uint32_t num_colors, int max_iters, int num_bits, uint32_t *colortable,
                               dq_split_record *records, double *cluster_mean, uint32_t *cluster_size);

/* Unique colours and counts of host pixels, in unspecified order. Returns U. Capacity numPixels each. */
uint32_t dq_debug_histogram(dq_context *ctx, const uint32_t *inPixels, uint32_t numPixels, uint32_t *colours,
                            uint32_t *counts);

/* Tracing aid for the persistent split kernel: when enabled, CTA 0 records (tag<<32|arg, SM clock) pairs at
 * its phase boundaries during the next calls.  Call again with pairs_out to fetch the last trace
 * (returns the number of pairs).  Tags: 1 round begin, 2 children finalised, 3 replay done, 4 jobs
 * issued, 5 barrier after controller, 6 pass done, 7 partition done, 8 root statistics done, 9 kernel entered,
 * 10 histogram collected, 11 root sums reduced, 12 root barrier passed, 13 narrow job done (arg = its passes,
 * the final one included). */
uint32_t dq_debug_split_timeline(dq_context *ctx, int enable, uint64_t *pairs_out, uint32_t capacity_pairs);

/* Host-only pieces of the path (no device needed): the palette handling the shim does between the
 * kernels, exposed so that CPU-only tests can check it against the oracle.
 *   dq_host_dedup_palette       first occurrence wins, order kept (quant_util.cpp:93-118); returns the new size.
 *   dq_host_build_search_tables sorted palette (the reference's std::sort by r+g+b) and lut_init[766]
 *                               (DivQuantMapColors.cpp:267-383).
 *   dq_host_build_label_table   for each position s of that sorted palette, the caller's index of the last entry with
 *                               that 24-bit colour: the per-item table the batch remap reads for labels. */
uint32_t dq_host_dedup_palette(uint32_t *colortable, uint32_t num_colors);
void dq_host_build_search_tables(const uint32_t *colortable, int num_colors, uint32_t *sorted_out, int32_t *lut_init_out);
void dq_host_build_label_table(const uint32_t *colortable, int num_colors, uint32_t *labels_out);
/* Host logic of the re-split with forced cuts (dq_call_stats::cut_overrides): of n <= 16 flagged cut entries, each a range
 * [begin, begin + size) of point positions with the resolver's status (3 = the reference cuts this node elsewhere), which
 * ones are forced in the next run -- the status-3 entries whose range does not lie inside another status-3 entry's, while
 * fewer than 16 cuts are forced in all (`already` = those forced by earlier runs).  Writes their indices to picked_out,
 * returns how many. */
uint32_t dq_host_select_cut_overrides(const uint32_t *begin, const uint32_t *size, const uint32_t *status, uint32_t n,
                                      uint32_t already, uint32_t *picked_out);

const char *dq_version(void);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif

#ifdef __cplusplus
}
#endif
#endif /* DIVQUANT_B200_H */

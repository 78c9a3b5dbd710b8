// dq_context.cu -- host side of libdivquant_b200.so: contexts, buffer management, the pipeline
// that strings the kernels together, and the extern "C" layer of include/divquant_b200.h.
//
// Pipeline of quant_recurse (reference: DivQuant/quant_util.cpp:20-158):
//   H2D pixels -> hist_insert (or points_from_pixels when allPixelsUnique)
//              -> split kernel (persistent, cooperative; collects the histogram in its first pass; small inputs
//                 leave into the ordered path)                                   = quant_varpart_fast
//              -> palette to the host (mapped mailbox the kernel writes last; else two small copies);
//                 host: drop empty/duplicate entries, std::sort by r+g+b, lut_init
//              -> map_unique (tables in its parameter block for K <= 256) + map_gather, or map_pixels (brute force)
//              -> D2H pixels
// Streams of frames go through dq_pipeline: several such chains side by side, one lane (context + host thread) each.
// The product has no CPU path for any per-pixel or per-point work; the host only handles the <= K
// palette words exactly as the reference's scalar code does.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <mutex>
#include <set>
#include <thread>
#include <vector>

#include "../../include/divquant_b200.h"
#include "dq_kernels.cuh"
#include "dq_map_int.cuh"
#include "dq_split.cuh"

namespace {

using namespace dq;

template <typename T>
struct DevBuf {
  T *ptr = nullptr;
  size_t cap = 0;
  void ensure(size_t n) {
    if (n <= cap) return;
    if (ptr) DQ_CUDA_CHECK(cudaFree(ptr));
    size_t want = n + n / 8 + 64;  // grow with slack so that slowly growing inputs do not realloc
    DQ_CUDA_CHECK(cudaMalloc(&ptr, want * sizeof(T)));
    cap = want;
  }
  void release() {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
  }
};

// Small control block shared with the kernels (one allocation, one memset per call).
struct ControlBlock {
  uint32_t ucount;
  uint32_t pad0[3];
  uint64_t root_acc[kAccWords];
  uint32_t ctl[kCtlWords];
  unsigned int barrier;
  uint32_t pad1[3];
  uint32_t result[4];
};

// Reference Pixel_Int (DivQuantHeader.h:40-44): element type handed to std::sort, kept identical in
// layout so that libstdc++'s introsort produces the reference's permutation of equal sums.
struct PaletteEntry {
  int red, green, blue;
  int weight;
};
inline bool palette_less(const PaletteEntry &a, const PaletteEntry &b) { return a.weight < b.weight; }

constexpr int kLutEntries = 3 * 255 + 1;
static_assert(kLutEntries == kBatchLutEntries, "lut_init of the batch remap");

// Pinned host staging that grows like DevBuf.
struct PinnedBuf {
  uint32_t *ptr = nullptr;
  size_t cap = 0;
  void ensure(size_t n) {
    if (n <= cap) return;
    if (ptr) DQ_CUDA_CHECK(cudaFreeHost(ptr));
    const size_t want = n + n / 8 + 64;
    DQ_CUDA_CHECK(cudaMallocHost(&ptr, want * sizeof(uint32_t)));
    cap = want;
  }
  void release() {
    if (ptr) cudaFreeHost(ptr);
    ptr = nullptr;
    cap = 0;
  }
};

}  // namespace

struct dq_context {
  int device = 0;
  int sm_count = 0;
  int split_ctas = 0;  // CTAs of the persistent split kernel (<= sm_count); fewer leaves SMs to concurrent contexts
  cudaStream_t stream = nullptr;
  uint32_t *d_table = nullptr;  // 2^24 counters, all zero between calls (hist_collect zeroes what it reads)
  uint32_t *d_map = nullptr;    // 2^24 mapped colours; only entries written by the current call are ever read, never cleared
  ControlBlock *d_cb = nullptr;
  ControlBlock *h_cb = nullptr;  // pinned
  DevBuf<uint32_t> d_in, d_out, d_uniq;
  DevBuf<uint2> d_pts0, d_pts1;
  DevBuf<uint2> d_flat;         // large tie resolver: the points by position
  DevBuf<uint32_t> d_sortvals;  // ... and the payload of its sort
  DevBuf<uint32_t> d_ovr;       // cuts taken from the resolver (SplitArgs::cut_overrides) of the call in flight
  DevBuf<uint64_t> d_keys;
  // sized by K
  DevBuf<SplitNode> d_nodes;
  DevBuf<SplitJob> d_jobs;
  DevBuf<uint64_t> d_acc;
  DevBuf<int32_t> d_ctl_i32;
  DevBuf<double> d_ctl_f64;
  DevBuf<uint32_t> d_palette, d_cluster_size, d_sorted;
  DevBuf<double> d_cluster_mean;
  DevBuf<SplitRecord> d_records;
  DevBuf<int4> d_pal_scratch;
  DevBuf<unsigned long long> d_timeline;
  DevBuf<unsigned long long> d_slots;
  DevBuf<uint32_t> d_progress;
  int exact_small = 1;    // small weighted inputs take the sequential-order kernel (DIVQUANT_B200_EXACT_SMALL=0 turns it off)
  uint32_t exact_max_points = kExactDefaultPoints;  // ... up to this many unique colours (DIVQUANT_B200_EXACT_MAX)
  DevBuf<uint64_t> d_exact;
  DevBuf<uint32_t> d_tie;  // flagged clusters / nodes, resolver status words, a counter (layout: dq_split.cuh, kTieListWords)
  // A quantize call between its two halves (quantize_begin / quantize_finish): the one description of its split, from
  // which every run of the split kernel takes its inputs and outputs (run_split).
  struct QuantState {
    uint32_t n = 0, rows = 0, cols = 0, K = 0, point_cap = 0;
    const uint32_t *d_in = nullptr;
    int num_bits = 8, dec = 1, max_iters = 10;
    double norm = 0.0;
    // the points are a histogram (of the sampled pixels of d_in, or of the merged lists): weighted, collected by the split
    // kernel's first pass, and a unique list of them stays in d_uniq for a table remap.  Otherwise they are in d_pts0.
    bool table_dirty = false;
    dq_split_record *records = nullptr;
    double *mean_out = nullptr;
    uint32_t *size_out = nullptr;
    // the paths of the call, fixed before its first run (plan_paths)
    bool v2 = false;        // the latency-optimised split kernel (K <= kSplit2MaxColors); else the generic one
    bool audited = false;   // the split audits its decisions against the reference's rounding noise (dq_tie.cuh)
    bool report_unaudited = false;  // weighted and not audited: a run beyond its ordered-path limit reports kTieUnaudited
    uint32_t exact_limit = 0;  // points up to which a run takes the ordered path (0: never); the ordered re-run: kExactMaxPoints
    bool mailbox = false;   // the palette comes back through the mapped mailbox (else stream wait + copies)
    bool resolve_ok = false;  // a flagged frame may go to the tie resolver (quantize_step checks its flags and lists)
    bool rerun_ok = false;    // ... or be computed again on the ordered path (if it has at most kExactMaxPoints points)
    SplitArgs split;          // the split launched last, whose palette run_split_finish collects
    enum class Step { kSplit, kResolve, kResolveLarge, kOrdered } step = Step::kSplit;  // what quantize_step waits for next
    uint32_t flags = 0, flags_all = 0, tie_count = 0, cut_count = 0, k_first = 0, resplits = 0;
    CutOverride h_ovr[kCutOverrideCap];  // forced cuts of the next run (SplitRun::kForcedCuts)
    uint32_t n_ovr = 0;
    // row-sharded call (dq_rows): the histogram and the first-seen indexes come from the gathered per-shard lists, not
    // from pixels, and there is no ordered re-run (that needs the whole image in order)
    struct Merged {
      const uint32_t *colours = nullptr, *counts = nullptr, *first = nullptr;  // [world][cap], [world][cap], [world][cap + 1]
      uint32_t cap = 0, world = 0;
    } merged;
  } qs;
  cudaEvent_t tie_ev = nullptr;
  // Tie audit of the exact-integer split (dq_tie.cuh): 0 = off, 1 = report in dq_call_stats::tie_flags only,
  // 2 (default) = a flagged frame is computed again in the reference's summation order (DIVQUANT_B200_TIE)
  int tie_policy = 2;
  int resolve_mode = 3;  // bit 0: the resolver's shared-memory form, bit 1: its large form (DIVQUANT_B200_RESOLVE; testing)
  long long spin_cycles = 0;  // DIVQUANT_B200_SPIN_MS: bound of the split kernel's waits on other CTAs (0 = built-in 0.2 s)
  int trace_split = 0;
  int profile_narrow = 0;  // DQ_PROFILE_NARROW set: the cycle counters of a -DDQ_PROFILE_NARROW build to stderr after every split
  int *d_lut = nullptr;
  // pinned staging for the palette-sized transfers
  uint32_t *h_small = nullptr;
  size_t h_small_words = 0;
  dq_call_stats stats;
  int display_timings = 1;
  int profiling = 0;
  cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  void mark(int i) {
    if (profiling) DQ_CUDA_CHECK(cudaEventRecord(ev[i], stream));
  }
  // Host waits on the hot path.  Default: spin (lowest latency).  blocking_wait: the thread sleeps on an event, which
  // is what a frame pipeline with more lanes than free host cores wants.
  int blocking_wait = 0;
  cudaEvent_t wait_ev = nullptr;
  // host mailbox of the split kernel (mapped pinned memory, SplitArgs::mailbox)
  volatile uint32_t *mailbox = nullptr;
  uint32_t mailbox_seq = 0;
  // quant_recurse over a batch of items (dq_batch.cu; quant_recurse_batch below)
  DevBuf<uint32_t> b_work;    // [items | per-item results | palettes | histogram slices: colours, counts, first seen]
  DevBuf<uint32_t> b_tables;  // [remap tiles | per-item (offset, size) | sorted palettes | lut_init, label tables as uint16]
  DevBuf<uint32_t> b_labels;  // label image of dq_map_colors_batch_ctx
  DevBuf<uint32_t> b_cluster_size;
  DevBuf<double> b_cluster_mean;
  PinnedBuf b_up, b_down, b_tab;
  dq_batch_stats batch_stats = {};
  // quant_recurse of every region of a tag image (dq_regions.cu; quant_regions_impl below): the sort's (tag, index) pairs
  // (2 x n, ping-pong), the pixels in sorted order [in | out | labels], [per-tile digit counts | digit totals | offsets]
  DevBuf<uint2> r_pairs;
  DevBuf<uint32_t> r_px, r_scratch;
  PinnedBuf r_offsets;
  void wait() {
    if (!blocking_wait) {
      DQ_CUDA_CHECK(cudaStreamSynchronize(stream));
      return;
    }
    if (!wait_ev) DQ_CUDA_CHECK(cudaEventCreateWithFlags(&wait_ev, cudaEventBlockingSync | cudaEventDisableTiming));
    DQ_CUDA_CHECK(cudaEventRecord(wait_ev, stream));
    DQ_CUDA_CHECK(cudaEventSynchronize(wait_ev));
  }

  void ensure_small(size_t words) {
    if (words <= h_small_words) return;
    if (h_small) DQ_CUDA_CHECK(cudaFreeHost(h_small));
    DQ_CUDA_CHECK(cudaMallocHost(&h_small, words * sizeof(uint32_t)));
    h_small_words = words;
  }
};

namespace {

void require_device(dq_context *ctx) { DQ_CUDA_CHECK(cudaSetDevice(ctx->device)); }

// ---- host handling of the <= K palette words ------------------------------------------------------

// First occurrence of each word survives, order kept (quant_util.cpp:93-118).
uint32_t dedup_palette(uint32_t *colortable, uint32_t n) {
  if (n <= 1) return n;
  uint32_t cap = 16;
  while (cap < 4 * n) cap <<= 1;
  std::vector<uint32_t> slots(cap, 0xFFFFFFFFu);  // palette words have a zero alpha byte, so all-ones is free
  uint32_t kept = 0;
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t w = colortable[i];
    uint32_t h = (w * 2654435761u) & (cap - 1);
    bool seen = false;
    while (slots[h] != 0xFFFFFFFFu) {
      if (slots[h] == w) {
        seen = true;
        break;
      }
      h = (h + 1) & (cap - 1);
    }
    if (!seen) {
      slots[h] = w;
      colortable[kept++] = w;
    }
  }
  return kept;
}

// Sorted palette + start-index table of map_colors_mps (DivQuantMapColors.cpp:267-383).
void build_search_tables(const uint32_t *colortable, int n, uint32_t *sorted_out, int *lut_out) {
  std::vector<PaletteEntry> v((size_t)n);
  for (int i = 0; i < n; ++i) {
    const uint32_t p = colortable[i];
    v[i].blue = (int)(p & 0xFF);
    v[i].green = (int)((p >> 8) & 0xFF);
    v[i].red = (int)((p >> 16) & 0xFF);
    v[i].weight = v[i].red + v[i].green + v[i].blue;
  }
  std::sort(v.begin(), v.end(), palette_less);
  for (int i = 0; i < n; ++i)
    sorted_out[i] = ((uint32_t)v[i].red << 16) | ((uint32_t)v[i].green << 8) | (uint32_t)v[i].blue;
  int low = (n >= 2) ? (int)(0.5 * (v[0].weight + v[1].weight) + 0.5) : 1;
  for (int k = 0; k < low; ++k) lut_out[k] = 0;
  int high = (n >= 2) ? (int)(0.5 * (v[n - 2].weight + v[n - 1].weight) + 0.5) : 1;
  for (int k = high; k < kLutEntries; ++k) lut_out[k] = n - 1;
  for (int ic = 1; ic < n - 1; ++ic) {
    low = (int)(0.5 * (v[ic - 1].weight + v[ic].weight) + 0.5);
    high = (int)(0.5 * (v[ic].weight + v[ic + 1].weight) + 0.5);
    for (int k = low; k < high; ++k) lut_out[k] = ic;
  }
}

// For every entry of the sorted palette of build_search_tables, the caller's index of the LAST palette entry with that
// 24-bit colour: the label mapQuantPixelsToColortableIndexes gives a pixel mapped to it (it fills an unordered_map in
// palette order, OpenCVUtil.cpp:795-799).
void build_label_table(const uint32_t *colortable, int n, const uint32_t *sorted, uint32_t *labels_out) {
  std::vector<uint64_t> keyed((size_t)n);  // (colour, index): ascending colour, then ascending index
  for (int i = 0; i < n; ++i) keyed[i] = ((uint64_t)(colortable[i] & 0x00FFFFFFu) << 32) | (uint32_t)i;
  std::sort(keyed.begin(), keyed.end());
  for (int s = 0; s < n; ++s) {
    const uint64_t past = ((uint64_t)sorted[s] + 1) << 32;  // every sorted entry is in the palette: the one before is its last
    labels_out[s] = (uint32_t)*(std::lower_bound(keyed.begin(), keyed.end(), past) - 1);
  }
}

// ---- device pipeline stages -----------------------------------------------------------------------

void reset_control(dq_context *ctx) {
  DQ_CUDA_CHECK(cudaMemsetAsync(ctx->d_cb, 0, sizeof(ControlBlock), ctx->stream));
}

// Which run of a quantize call's split: the first, the ordered re-run of a flagged frame (every input the ordered path
// can hold goes there), or the re-run with the resolver's forced cuts (QuantState::h_ovr).
enum class SplitRun { kFirst, kOrdered, kForcedCuts };

// Decides, once before the first run of the call that ctx->qs describes, the paths that stay fixed for the whole call:
// the split kernel, its tie audit, the ordered path's limit, how the palette comes back, and which recovery steps a
// flagged frame may take (quantize_step).
void plan_paths(dq_context *ctx) {
  dq_context::QuantState &q = ctx->qs;
  // a histogram is weighted; one of the pixels in q.d_in also gives the ordered path its input (a merged one has no
  // pixels here)
  const bool hist = q.table_dirty, pixels = hist && q.merged.colours == nullptr;
  const bool settle = ctx->tie_policy == 2 && hist && ctx->exact_small;
  q.v2 = q.K <= kSplit2MaxColors;
  q.audited = hist && q.v2 && ctx->tie_policy != 0;
  q.report_unaudited = hist && !q.audited && ctx->tie_policy != 0;
  q.exact_limit = 0;
  if (pixels && q.K <= kExactMaxColors && ctx->exact_small && ctx->exact_max_points > 0)
    // the generic kernel carries no tie audit: everything the ordered path can hold goes there
    q.exact_limit = (!q.v2 && ctx->tie_policy != 0) ? kExactMaxPoints : ctx->exact_max_points;
  q.mailbox = q.v2 && !ctx->blocking_wait && !ctx->trace_split && q.records == nullptr && q.mean_out == nullptr &&
              q.size_out == nullptr;
  q.resolve_ok = settle && q.records == nullptr && q.mean_out == nullptr;
  q.rerun_ok = settle && q.v2 && pixels;
}

// Queues the divisive phase that ctx->qs describes, on its points: the histogram in the direct table and d_uniq
// (q.table_dirty), or ctx->d_pts0[0..U).  U is read on the device from d_cb->ucount.  Nothing is waited for: the caller
// polls split_ready() and collects the palette with run_split_finish().
void run_split(dq_context *ctx, SplitRun run) {
  dq_context::QuantState &q = ctx->qs;
  const uint32_t K = q.K, point_capacity = q.point_cap;
  const int max_iters = q.max_iters;
  const bool hist = q.table_dirty;  // (collected by the split kernel)
  if (max_iters < 1 || max_iters > kSplitMaxIters) {
    fprintf(stderr, "divquant_b200: max_iters ( %d ) must be in [1,%d] (the reference hard-wires local k-means on)\n",
            max_iters, kSplitMaxIters);
    abort();
  }
  const uint32_t node_cap = 4 * K + 8;
  ctx->d_pts1.ensure(point_capacity);
  ctx->d_nodes.ensure(node_cap);
  ctx->d_jobs.ensure((size_t)2 * K);
  ctx->d_acc.ensure(split_acc_words(K, max_iters));
  ctx->d_ctl_i32.ensure((size_t)2 * K + node_cap + 16);
  ctx->d_ctl_f64.ensure((size_t)K + node_cap + 16);
  ctx->d_palette.ensure(K);
  ctx->d_cluster_size.ensure(K);
  ctx->d_cluster_mean.ensure((size_t)3 * K);
  if (q.records) ctx->d_records.ensure(K);

  SplitArgs a;
  memset(&a, 0, sizeof(a));
  a.pts[0] = ctx->d_pts0.ptr;
  a.pts[1] = ctx->d_pts1.ptr;
  a.num_points = 0;
  a.num_points_dev = &ctx->d_cb->ucount;
  a.num_colors = K;
  a.max_iters = max_iters;
  a.shift = 8 - q.num_bits;
  a.norm = q.norm;
  a.nodes = ctx->d_nodes.ptr;
  a.node_cap = node_cap;
  a.jobs = ctx->d_jobs.ptr;
  a.acc = ctx->d_acc.ptr;
  a.root_acc = ctx->d_cb->root_acc;
  a.ctl = ctx->d_cb->ctl;
  a.barrier = &ctx->d_cb->barrier;
  a.g_cluster_node = ctx->d_ctl_i32.ptr;
  a.g_cluster_tse = ctx->d_ctl_f64.ptr;
  a.palette = ctx->d_palette.ptr;
  a.result = ctx->d_cb->result;
  a.cluster_mean = ctx->d_cluster_mean.ptr;
  a.cluster_size = ctx->d_cluster_size.ptr;
  a.records = q.records ? ctx->d_records.ptr : nullptr;
  if (ctx->trace_split) {
    ctx->d_timeline.ensure(8192);
    DQ_CUDA_CHECK(cudaMemsetAsync(ctx->d_timeline.ptr, 0, sizeof(unsigned long long), ctx->stream));
    a.timeline = ctx->d_timeline.ptr;
    a.timeline_cap = 8192;
  }

  a.spin_cycles = ctx->spin_cycles;
  a.tie_audit = q.audited ? 1u : 0u;
  if (a.tie_audit) {
    ctx->d_tie.ensure(kTieListWords);
    a.tie_list = ctx->d_tie.ptr;
    if (run == SplitRun::kForcedCuts) {
      a.cut_overrides = reinterpret_cast<const CutOverride *>(ctx->d_ovr.ptr);
      a.num_cut_overrides = q.n_ovr;
    }
  }
  ctx->mark(2);
  // (the ordered re-run is only queued when q.rerun_ok, which implies every condition of q.exact_limit)
  const bool exact_path = run == SplitRun::kOrdered || q.exact_limit > 0;
  ExactSampling sampling;
  memset(&sampling, 0, sizeof(sampling));
  if (exact_path) {
    // small inputs: the reference's own summation order (dq_split_exact.cuh); large ones take one branch
    ctx->d_ctl_f64.ensure((size_t)8 * K + node_cap + 16);
    a.g_cluster_tse = ctx->d_ctl_f64.ptr;
    a.exact_small_max = run == SplitRun::kOrdered ? kExactMaxPoints : q.exact_limit;
    ctx->d_exact.ensure((split_exact_scratch_bytes() + ((size_t)8 * K + 16 + 64) * sizeof(uint32_t)) / 8 + 2);
    sampling = exact_sampling(q.d_in, q.rows, q.cols, (uint32_t)q.dec, q.num_bits);
  }
  if (q.v2) {
    Split2Extra x;
    memset(&x, 0, sizeof(x));
    const size_t slot_cap = split2_slot_capacity(point_capacity, K, ctx->sm_count);
    ctx->d_slots.ensure(2 * slot_cap * kAccWords);
    ctx->d_nodes.ensure((size_t)8 * K + 16);
    a.nodes = ctx->d_nodes.ptr;
    x.slots = ctx->d_slots.ptr;
    x.slot_cap = (uint32_t)slot_cap;
    ctx->d_progress.ensure(1024);
    x.progress = ctx->d_progress.ptr;
    x.collect_uniq = hist ? ctx->d_uniq.ptr : nullptr;
    x.collect_table = hist ? ctx->d_table : nullptr;
    if (ctx->profile_narrow) DQ_CUDA_CHECK(cudaMemsetAsync(ctx->d_progress.ptr, 0, 1024 * sizeof(uint32_t), ctx->stream));
    if (q.mailbox) {
      void *dev = nullptr;
      DQ_CUDA_CHECK(cudaHostGetDevicePointer(&dev, const_cast<uint32_t *>(ctx->mailbox), 0));
      a.mailbox = static_cast<uint32_t *>(dev);
      a.mailbox_seq = ++ctx->mailbox_seq;
      if (a.mailbox_seq == 0) a.mailbox_seq = ++ctx->mailbox_seq;  // 0 is the idle value
    }
    // the ordered path always runs inside this kernel: its plan makes room for it in the dynamic shared memory
    const SplitLaunch plan = split2_plan(ctx->split_ctas, ctx->sm_count, K);
    if (exact_path) {
      x.exact_fused = plan.grid > 1 ? 2 : 1;
      x.exact_src = sampling;
      x.exact_first_seen = ctx->d_map;
      x.exact_scratch = reinterpret_cast<unsigned char *>(ctx->d_exact.ptr);
      x.exact_f64 = ctx->d_ctl_f64.ptr;
      x.exact_i32 = ctx->d_ctl_i32.ptr;
    }
    split2_launch(a, x, plan, ctx->stream);
  } else {
    if (exact_path) {
      split_exact_launch(a, sampling, reinterpret_cast<unsigned char *>(ctx->d_exact.ptr), ctx->d_uniq.ptr, ctx->d_table, ctx->d_map, ctx->d_ctl_f64.ptr, ctx->d_ctl_i32.ptr, ctx->stream);
      ctx->stats.kernel_launches += 2;
    }
    if (hist) {  // the generic kernel has no fused collect
      hist_collect(ctx->d_uniq.ptr, &ctx->d_cb->ucount, point_capacity, ctx->d_table, ctx->d_pts0.ptr, true, ctx->sm_count, ctx->stream);
      ctx->stats.kernel_launches++;
    }
    split_launch(a, split_plan(std::min(ctx->split_ctas > 0 ? ctx->split_ctas : ctx->sm_count, ctx->sm_count), K), ctx->stream);
  }
  ctx->mark(3);
  ctx->stats.kernel_launches++;
  q.split = a;
}

// Has the split launched last on this context delivered its palette?  (non-blocking; true when there is nothing to poll)
bool split_ready(dq_context *ctx) {
  const SplitArgs &a = ctx->qs.split;
  if (a.mailbox == nullptr) return true;
  if (ctx->mailbox[0] == a.mailbox_seq) return true;
  return cudaStreamQuery(ctx->stream) != cudaErrorNotReady;  // an error exit leaves the stream idle without the number
}

// Collects the palette of the split launched last into colortable_out, and the records / means / sizes ctx->qs asks for.
// Returns the number of palette entries.
uint32_t run_split_finish(dq_context *ctx, uint32_t *colortable_out) {
  const dq_context::QuantState &q = ctx->qs;
  const SplitArgs &a = q.split;
  const uint32_t K = q.K;
  ctx->ensure_small((size_t)K + 16);
  bool mailed = false;
  if (a.mailbox != nullptr) {
    // The kernel's last act is to store palette, result and diagnostics into mapped host memory and then the sequence
    // number: poll for it instead of waiting for the stream to drain and two copies to come back.  If the stream is
    // found idle without the number (an error exit), fall through to the copies below.
    const uint32_t want = a.mailbox_seq;
    for (unsigned spins = 0;; ++spins) {
      if (ctx->mailbox[0] == want) {
        mailed = true;
        break;
      }
      if ((spins & 0xFFFu) == 0xFFFu && cudaStreamQuery(ctx->stream) != cudaErrorNotReady) {
        mailed = (ctx->mailbox[0] == want);
        break;
      }
    }
    if (mailed) {
      std::atomic_thread_fence(std::memory_order_acquire);
      ctx->h_cb->ucount = ctx->mailbox[1];
      for (int i = 0; i < 4; ++i) ctx->h_cb->result[i] = ctx->mailbox[2 + i];
      for (int i = 0; i < (int)kCtlWords; ++i) ctx->h_cb->ctl[i] = ctx->mailbox[6 + i];
      for (uint32_t i = 0; i < K; ++i) ctx->h_small[i] = ctx->mailbox[kMailboxPalette + i];
    }
  }
  if (!mailed) {
    DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->h_small, ctx->d_palette.ptr, K * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->h_cb, ctx->d_cb, sizeof(ControlBlock), cudaMemcpyDeviceToHost, ctx->stream));
    ctx->wait();
  }
  if (ctx->h_cb->ctl[kCtlError] != 0) {
    fprintf(stderr, "divquant_b200: split controller failed (code %u, kernel v%d, detail %u/%u/%u, barrier counter %u; internal error)\n",
            ctx->h_cb->ctl[kCtlError], q.v2 ? 2 : 1, ctx->h_cb->ctl[kCtlWords - 1], ctx->h_cb->ctl[kCtlJobs],
            ctx->h_cb->ctl[kCtlTiles], ctx->h_cb->ctl[kCtlNodes]);
    if (q.v2) {
      std::vector<uint32_t> prog(split2_max_ctas(ctx->sm_count, K));
      cudaMemcpy(prog.data(), ctx->d_progress.ptr, prog.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost);
      fprintf(stderr, "  last stage per CTA:");
      for (size_t i = 0; i < prog.size(); ++i) fprintf(stderr, " %u", prog[i]);
      fprintf(stderr, "\n");
    }
    abort();
  }
  if (q.v2 && ctx->profile_narrow) {
    uint32_t prof[8];
    cudaMemcpy(prof, ctx->d_progress.ptr + 756, sizeof(prof), cudaMemcpyDeviceToHost);
    uint32_t wp[9];
    cudaMemcpy(wp, ctx->d_progress.ptr + 764, sizeof(wp), cudaMemcpyDeviceToHost);
    if (wp[3])
      fprintf(stderr, "wide profile (cycles per job-pass, thread 0 of every participant): gather %.0f derive+sync %.0f classify+reduce+publish %.0f (classify %.0f, stage1+sync %.0f, stage2 %.0f, publish %.0f, closing barrier %.0f) ; %u job-passes\n",
              (double)wp[0] / wp[3], (double)wp[1] / wp[3], (double)wp[2] / wp[3], (double)wp[4] / wp[3], (double)wp[5] / wp[3],
              (double)wp[6] / wp[3], (double)wp[7] / wp[3], (double)wp[8] / wp[3], wp[3]);
    if (prof[4])
      fprintf(stderr, "narrow profile (cycles per pass, thread 0): classify %.0f stage1+sync %.0f warp0(stage2+derive) %.0f sync %.0f ; %u passes, %u points\n",
              (double)prof[0] / prof[4], (double)prof[1] / prof[4], (double)prof[2] / prof[4], (double)prof[3] / prof[4], prof[4], prof[5]);
  }
  const uint32_t actual = ctx->h_cb->result[0], empty = ctx->h_cb->result[1];
  memcpy(colortable_out, ctx->h_small, actual * sizeof(uint32_t));
  if (empty) fprintf(stderr, "# empty clusters: %d\n", (int)empty);  // (:1067-1070)
  ctx->stats.num_points = ctx->h_cb->ucount;
  ctx->stats.requested_colors = K;
  ctx->stats.actual_colors = actual;
  ctx->stats.empty_clusters = empty;
  ctx->stats.split_rounds = ctx->h_cb->ctl[kCtlRounds];
  ctx->stats.splits_computed = ctx->h_cb->ctl[kCtlSplits];
  ctx->stats.tie_flags = a.tie_audit ? ctx->h_cb->ctl[kCtlTie] : 0u;
  // exact-integer sums without an audit (the generic kernel beyond the ordered path's reach): say so
  if (q.report_unaudited && ctx->h_cb->ucount > a.exact_small_max) ctx->stats.tie_flags |= (uint32_t)kTieUnaudited;
  if (q.records && K > 1)
    DQ_CUDA_CHECK(cudaMemcpy(q.records, ctx->d_records.ptr, (size_t)(K - 1) * sizeof(SplitRecord), cudaMemcpyDeviceToHost));
  if (q.mean_out) DQ_CUDA_CHECK(cudaMemcpy(q.mean_out, ctx->d_cluster_mean.ptr, (size_t)3 * K * sizeof(double), cudaMemcpyDeviceToHost));
  if (q.size_out) DQ_CUDA_CHECK(cudaMemcpy(q.size_out, ctx->d_cluster_size.ptr, (size_t)K * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  return actual;
}

// The reference trusts numRows/numCols blindly (its sampling loop addresses inPixels[ic + ir*numRows],
// DivQuantMapColors.cpp:120-124); a stray index would be an illegal device address here, so refuse it.
void check_sampling(uint32_t n, uint32_t rows, uint32_t cols, uint32_t dec) {
  if (rows == 0 || cols == 0) {
    fprintf(stderr, "divquant_b200: numRows and numCols must be positive\n");
    abort();
  }
  const uint64_t last_r = ((uint64_t)(rows - 1) / dec) * dec, last_c = ((uint64_t)(cols - 1) / dec) * dec;
  if (last_c + last_r * rows >= n) {
    fprintf(stderr, "divquant_b200: sampling grid %u x %u (step %u) reaches beyond the %u input pixels\n", rows, cols, dec, n);
    abort();
  }
}

// Histogram of d_in into the table + unique list; leaves U in d_cb->ucount (device).
void run_histogram(dq_context *ctx, const uint32_t *d_in, uint32_t n, uint32_t rows, uint32_t cols, uint32_t dec, int bits) {
  check_sampling(n, rows, cols, dec);
  ctx->d_uniq.ensure(n);
  hist_insert(d_in, n, rows, cols, dec, bits, ctx->d_table, ctx->d_uniq.ptr, &ctx->d_cb->ucount, ctx->sm_count, ctx->stream,
              ctx->exact_small ? ctx->d_map : nullptr);
  ctx->stats.kernel_launches++;
}

void upload_search_tables(dq_context *ctx, const uint32_t *colortable, int k) {
  ctx->ensure_small((size_t)k + kLutEntries + 16);
  uint32_t *h_sorted = ctx->h_small;
  int *h_lut = reinterpret_cast<int *>(ctx->h_small + k);
  build_search_tables(colortable, k, h_sorted, h_lut);
  // sorted palette and start-index table travel in one copy: [k palette words | 766 lut entries]
  ctx->d_sorted.ensure((size_t)k + kLutEntries);
  ctx->d_lut = reinterpret_cast<int *>(ctx->d_sorted.ptr + k);
  (void)h_lut;
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_sorted.ptr, h_sorted, ((size_t)k + kLutEntries) * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                ctx->stream));
  // h_small is reused by later calls: the copies above must have been issued from it before then;
  // every caller synchronises the stream before returning.
}

void remap_bruteforce(dq_context *ctx, const uint32_t *d_in, uint32_t n, uint32_t *d_out, int k) {
  if (k > map_smem_palette_limit()) ctx->d_pal_scratch.ensure(k);
  ctx->mark(4);
  map_pixels(d_in, n, d_out, ctx->d_sorted.ptr, k, ctx->d_lut, ctx->d_pal_scratch.ptr, ctx->sm_count, ctx->stream);
  ctx->mark(5);
  ctx->mark(6);
  ctx->mark(7);
  ctx->stats.kernel_launches += (k > map_smem_palette_limit()) ? 2 : 1;
  ctx->stats.remap_path = 1;
}

// Table path: requires the unique list of exactly these pixels in d_uniq / d_cb->ucount.
void remap_through_table(dq_context *ctx, const uint32_t *d_in, uint32_t n, uint32_t *d_out, int k, uint32_t u_hint) {
  if (k > map_smem_palette_limit()) ctx->d_pal_scratch.ensure(k);
  ctx->mark(4);
  map_unique(ctx->d_uniq.ptr, &ctx->d_cb->ucount, u_hint, ctx->d_map, ctx->d_sorted.ptr, k, ctx->d_lut, ctx->d_pal_scratch.ptr,
             ctx->sm_count, ctx->stream);
  ctx->mark(5);
  map_gather(d_in, n, d_out, ctx->d_map, ctx->sm_count, ctx->stream);
  ctx->mark(6);
  ctx->mark(7);
  ctx->stats.kernel_launches += (k > map_smem_palette_limit()) ? 3 : 2;
  ctx->stats.remap_path = 2;
}

double sample_norm(uint32_t rows, uint32_t cols, int dec) {
  // norm_factor of calc_color_table (:172) == get_double_scale (:215) when rows = 1, dec = 1
  return 1.0 / (std::ceil(rows / (double)dec) * std::ceil(cols / (double)dec));
}

void check_quant_args(uint32_t n, uint32_t k, int num_bits) {
  if (!dq_validate_num_bits((unsigned char)num_bits)) abort();  // assert(0) in the reference (:1115-1118)
  if (n == 0 || k == 0) {
    fprintf(stderr, "divquant_b200: numPixels and the requested number of clusters must be positive\n");
    abort();  // assert(num_points > 0) / assert(num_colors > 0) (:249, :266)
  }
}

// The merged histogram of a row-sharded image in the direct table, and the whole image's first-seen index of every colour
// in d_map (what the resolver reads); leaves U in d_cb->ucount.
void run_merge(dq_context *ctx, const dq_context::QuantState::Merged &m) {
  hist_merge(m.colours, m.counts, m.world * m.cap, ctx->d_table, ctx->d_uniq.ptr, &ctx->d_cb->ucount, ctx->sm_count, ctx->stream,
             ctx->d_map);
  hist_merge_first(m.colours, m.counts, m.first, m.cap, m.world, ctx->d_map, ctx->sm_count, ctx->stream);
  ctx->stats.kernel_launches += 2;
}

// Control block cleared and the histogram of ctx->qs's source built again: the sampled pixels of q.d_in or, in a
// row-sharded call (whose other shards' pixels are not here), the gathered lists.  Leaves U in d_cb->ucount.
void rebuild_histogram(dq_context *ctx) {
  const dq_context::QuantState &q = ctx->qs;
  reset_control(ctx);
  if (q.merged.colours != nullptr) run_merge(ctx, q.merged);
  else run_histogram(ctx, q.d_in, q.n, q.rows, q.cols, (uint32_t)q.dec, q.num_bits);
}

// Queues the first run of the quantize call that the caller has described in ctx->qs: the points (the histogram of its
// source, or one per pixel of q.d_in), then the split.  Nothing is waited for.
void quantize_launch(dq_context *ctx) {
  const dq_context::QuantState &q = ctx->qs;
  plan_paths(ctx);
  ctx->mark(0);
  ctx->d_pts0.ensure(q.point_cap);
  if (q.table_dirty) {
    rebuild_histogram(ctx);
    ctx->mark(1);
  } else {
    reset_control(ctx);
    ctx->mark(1);
    points_from_pixels(q.d_in, q.n, ctx->d_pts0.ptr, ctx->sm_count, ctx->stream);
    ctx->stats.kernel_launches++;
    ctx->h_cb->ucount = q.n;
    DQ_CUDA_CHECK(cudaMemcpyAsync(&ctx->d_cb->ucount, &ctx->h_cb->ucount, sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  }
  run_split(ctx, SplitRun::kFirst);
}

// quant_varpart_fast on device-resident pixels.  First half: histogram (or points) and the split kernel are queued;
// nothing is waited for.
void quantize_begin(dq_context *ctx, uint32_t n, const uint32_t *d_in, uint32_t rows, uint32_t cols, uint32_t K, int num_bits,
                    int dec, int max_iters, int all_unique, dq_split_record *records, double *mean_out, uint32_t *size_out) {
  check_quant_args(n, K, num_bits);
  dq_context::QuantState &q = ctx->qs;
  q = dq_context::QuantState();
  q.n = n, q.rows = rows, q.cols = cols, q.K = K, q.d_in = d_in;
  q.num_bits = num_bits, q.dec = dec, q.max_iters = max_iters;
  q.records = records, q.mean_out = mean_out, q.size_out = size_out;
  if (all_unique && num_bits == 8 && dec == 1) {
    // uniform weight: every pixel is a point (DivQuantCluster.cpp:1130-1132)
    q.point_cap = n;
    q.norm = sample_norm(1, n, 1);
  } else {
    if (dec <= 0) {
      fprintf(stderr, "Decimation factor ( %d ) should be positive !\n", dec);
      abort();  // the reference dereferences the NULL it gets back (:1136); fail loudly instead
    }
    q.point_cap = ((rows + dec - 1) / dec) * ((cols + dec - 1) / dec);
    q.norm = sample_norm(rows, cols, dec);
    q.table_dirty = true;
  }
  quantize_launch(ctx);
}

// Second half, as a small state machine so that a host thread that drives several contexts never has to wait inside it
// (QuantState::step is what comes next):
//   kSplit         the split's palette is collected; a clean frame is done.  A flagged frame (tie audit, dq_tie.cuh) gets
//                  the resolver queued (only palette roundings and cuts in doubt: dq_resolve.cu) -> kResolve or
//                  kResolveLarge, or goes to the fallback
//   kResolve       the resolver's verdict: palette words patched, done -- or a cut the reference makes elsewhere: the split
//   kResolveLarge  once more with that cut forced -> kSplit -- or, after the shared-memory form, a chain through a large
//                  node: the large form -> kResolveLarge -- or the fallback
//   kOrdered       the ordered re-run's palette is collected, done
// The fallback queues the ordered re-run -> kOrdered where the call allows it and the ordered path holds the frame; else
// the frame is done and stays flagged in the stats.
// quantize_step() advances one step and says what to poll next; quantize_pending_ready() is the non-blocking poll.
enum QuantStepResult { kQuantDone = 0, kQuantPending = 1 };

// Which of the resolver's cut entries become forced cuts of the next run of the split (host logic of the re-split, pure):
// those the resolver found the reference cuts elsewhere (status 3) whose range of positions is not inside another such
// entry's -- a cut below a cut that changes is decided by the next run -- as long as there is room.  Appends to
// out[*n_out..cap) and returns how many it added.
uint32_t select_cut_overrides(const CutOverride *rec, const uint32_t *status, uint32_t n, CutOverride *out, uint32_t *n_out,
                              uint32_t cap) {
  uint32_t added = 0;
  for (uint32_t i = 0; i < n; ++i) {
    if (status[i] != 3u) continue;
    bool nested = false;
    for (uint32_t j = 0; j < n; ++j)
      nested = nested || (j != i && status[j] == 3u && rec[j].begin <= rec[i].begin &&
                          rec[i].begin + rec[i].size <= rec[j].begin + rec[j].size && (rec[j].size > rec[i].size || j < i));
    if (nested || *n_out >= cap) continue;
    out[(*n_out)++] = rec[i];
    ++added;
  }
  return added;
}

bool quantize_pending_ready(dq_context *ctx) {
  using Step = dq_context::QuantState::Step;
  if (ctx->qs.step == Step::kResolve || ctx->qs.step == Step::kResolveLarge)
    return cudaEventQuery(ctx->tie_ev) != cudaErrorNotReady;
  return split_ready(ctx);
}

QuantStepResult quantize_step(dq_context *ctx, uint32_t *k_inout, uint32_t *colortable) {
  using Step = dq_context::QuantState::Step;
  dq_context::QuantState &q = ctx->qs;
  const uint32_t K = q.K;
  auto rerun_or_done = [&]() {
    // Some decision of the exact-integer split sits inside the rounding noise of the reference's sequential sums:
    // the reference's own summation order decides.  The count table is all-zero again (the split kernel zeroed what
    // it collected), so the frame simply goes through the histogram and the split once more, on the ordered path.
    // Where the call or the frame's size rules that out, the frame is done and stays flagged in the stats.
    if (!q.rerun_ok || ctx->stats.num_points > kExactMaxPoints) return kQuantDone;
    rebuild_histogram(ctx);
    run_split(ctx, SplitRun::kOrdered);
    q.step = Step::kOrdered;
    return kQuantPending;
  };
  auto queue_resplit = [&]() {
    // The reference cuts some node on the other side of an integer than the exact mean does (the resolver found out, and
    // what the reference's mean is): the exact-integer split runs again with that node cut where the reference cuts it
    // (SplitArgs::cut_overrides).  Everything outside the node's subtree comes out as before.
    ctx->d_ovr.ensure(kCutOverrideCap * sizeof(CutOverride) / sizeof(uint32_t));
    DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_ovr.ptr, q.h_ovr, q.n_ovr * sizeof(CutOverride), cudaMemcpyHostToDevice, ctx->stream));
    rebuild_histogram(ctx);
    run_split(ctx, SplitRun::kForcedCuts);
    q.resplits++;
    q.step = Step::kSplit;
  };
  auto queue_resolve = [&](bool large) {
    // the resolver (dq_resolve.cu) in its shared-memory form, or its large form: chains through nodes of any size, a global
    // sort instead of one in shared memory; its verdict comes back in h_small: [palette | status words | reference cuts]
    const uint32_t U = ctx->stats.num_points;
    uint32_t n_pow2 = 2;
    while (n_pow2 < U) n_pow2 <<= 1;
    if (large) {
      ctx->d_keys.ensure(n_pow2);
      ctx->d_sortvals.ensure(n_pow2);
      ctx->d_flat.ensure(U);
    }
    uint32_t *d_status = ctx->d_tie.ptr + kTieStatus;
    DQ_CUDA_CHECK(cudaMemsetAsync(d_status, 0, 2 * kTieListCap * sizeof(uint32_t), ctx->stream));
    uint2 *pts[2] = {ctx->d_pts0.ptr, ctx->d_pts1.ptr};
    if (large) {
      tie_resolve_big_launch(ctx->d_nodes.ptr, ctx->h_cb->ctl[kCtlNodes], pts, ctx->d_map, U, q.norm, 8 - q.num_bits, ctx->d_tie.ptr,
                             q.tie_count, q.cut_count, ctx->d_keys.ptr, ctx->d_sortvals.ptr, ctx->d_flat.ptr,
                             ctx->d_tie.ptr + kTieCounter, ctx->d_palette.ptr, d_status, ctx->sm_count, ctx->stream);
      uint32_t steps = 0;
      for (uint32_t k = 2; k <= n_pow2; k <<= 1) steps += (uint32_t)__builtin_ctz(k);
      ctx->stats.kernel_launches += 3 + steps;
    } else {
      tie_resolve_launch(ctx->d_nodes.ptr, ctx->h_cb->ctl[kCtlNodes], pts, ctx->d_map, q.norm, 8 - q.num_bits, ctx->d_tie.ptr,
                         q.tie_count, q.cut_count, ctx->d_palette.ptr, d_status, ctx->stream);
      ctx->stats.kernel_launches++;
    }
    DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->h_small + K, d_status, (q.tie_count + q.cut_count) * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                                  ctx->stream));
    if (q.cut_count)
      DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->h_small + K + 2 * kTieListCap, ctx->d_tie.ptr + kTieRefCut, q.cut_count * sizeof(CutOverride),
                                    cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->h_small, ctx->d_palette.ptr, (size_t)q.k_first * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                                  ctx->stream));
    DQ_CUDA_CHECK(cudaEventRecord(ctx->tie_ev, ctx->stream));
    q.step = large ? Step::kResolveLarge : Step::kResolve;
  };
  if (q.step == Step::kSplit) {
    *k_inout = run_split_finish(ctx, colortable);
    q.flags = ctx->stats.tie_flags;
    q.flags_all |= q.flags;
    ctx->stats.tie_flags = q.flags_all;  // (a frame that needed forced cuts stays marked as flagged)
    ctx->stats.cut_overrides = q.n_ovr;
    if (q.flags == 0u) return kQuantDone;
    if (q.resolve_ok && (q.flags & ~(uint32_t)(kTieRound | kTieCut)) == 0u) {
      // Palette roundings and cuts are in doubt, nothing else (by far the commonest flags): both hang on the mean of ONE node,
      // which the resolver recomputes in the reference's arithmetic (dq_resolve.cu) on top of a first-seen pass over the pixels.
      // A rounding is rewritten; a cut either separates the same points as the reference's (nothing to do) or it does not
      // (status 3: the frame has to be computed again).
      q.tie_count = ctx->h_cb->ctl[kCtlTieCount];
      q.cut_count = ctx->h_cb->ctl[kCtlCutCount];
      if (q.tie_count + q.cut_count >= 1 && q.tie_count <= kTieListCap && q.cut_count <= kTieListCap && ctx->resolve_mode != 0) {
        if (q.merged.colours == nullptr) {  // (a merged histogram brought its first-seen indexes along: run_merge)
          first_seen_launch(exact_sampling(q.d_in, q.rows, q.cols, (uint32_t)q.dec, q.num_bits), ctx->d_map, ctx->stream);
          ctx->stats.kernel_launches++;
        }
        ctx->ensure_small((size_t)K + 16 + 8 * kTieListCap + 2);
        q.k_first = *k_inout;
        if (!ctx->tie_ev) DQ_CUDA_CHECK(cudaEventCreateWithFlags(&ctx->tie_ev, cudaEventDisableTiming));
        queue_resolve((ctx->resolve_mode & 1) == 0);
        return kQuantPending;
      }
    }
    return rerun_or_done();
  }
  if (q.step == Step::kOrdered) {
    *k_inout = run_split_finish(ctx, colortable);
    ctx->stats.tie_flags = q.flags;
    ctx->stats.ordered_rerun = 1;
    return kQuantDone;
  }
  // the resolver's verdict (kResolve, kResolveLarge)
  DQ_CUDA_CHECK(cudaEventSynchronize(ctx->tie_ev));  // (already complete when the caller polled)
  bool resolved = true, differs = false;
  for (uint32_t i = 0; i < q.tie_count + q.cut_count; ++i) {
    resolved = resolved && ctx->h_small[K + i] == 1u;
    differs = differs || ctx->h_small[K + i] == 3u;  // a cut the reference makes elsewhere: only a re-run helps
  }
  if (resolved) {
    memcpy(colortable, ctx->h_small, (size_t)q.k_first * sizeof(uint32_t));
    *k_inout = q.k_first;
    ctx->stats.tie_resolved = q.tie_count + q.cut_count;
    return kQuantDone;
  }
  if (differs && q.resplits < 8) {
    // status-3 cut entries whose range is not inside another one's (a cut below a cut that changes is decided next time)
    CutOverride rec[kTieListCap];  // (copied out: K odd leaves the doubles inside h_small unaligned)
    memcpy(rec, ctx->h_small + K + 2 * kTieListCap, q.cut_count * sizeof(CutOverride));
    const uint32_t *st = ctx->h_small + K + q.tie_count;
    const uint32_t added = select_cut_overrides(rec, st, q.cut_count, q.h_ovr, &q.n_ovr, kCutOverrideCap);
    if (added) {
      queue_resplit();
      return kQuantPending;
    }
  }
  if (q.step == Step::kResolve && !differs && (ctx->resolve_mode & 2)) {  // a chain through a large node: the large form
    queue_resolve(true);
    return kQuantPending;
  }
  return rerun_or_done();
}

// Blocking form.  Returns true if a unique list exists (d_uniq / d_cb->ucount) for a following table remap.
bool quantize_finish(dq_context *ctx, uint32_t *k_inout, uint32_t *colortable) {
  while (quantize_step(ctx, k_inout, colortable) != kQuantDone) {
  }
  return ctx->qs.table_dirty;
}

bool quantize_device(dq_context *ctx, uint32_t n, const uint32_t *d_in, uint32_t rows, uint32_t cols, uint32_t *k_inout,
                     uint32_t *colortable, int num_bits, int dec, int max_iters, int all_unique, dq_split_record *records,
                     double *mean_out, uint32_t *size_out) {
  quantize_begin(ctx, n, d_in, rows, cols, *k_inout, num_bits, dec, max_iters, all_unique, records, mean_out, size_out);
  return quantize_finish(ctx, k_inout, colortable);
}

// quant_recurse on device pixels in two halves, so that one host thread can keep several contexts busy: recurse_begin
// queues histogram + split; once split_ready(ctx), recurse_remap collects the palette, handles it exactly as the
// reference's host code does (duplicates, std::sort, lut_init) and queues the remap.  Neither waits for the GPU unless
// the tie audit flagged the frame.
void recurse_begin(dq_context *ctx, uint32_t n, const uint32_t *d_in, uint32_t K, int all_unique) {
  quantize_begin(ctx, n, d_in, 1, n, K, 8, 1, 10, all_unique, nullptr, nullptr, nullptr);
}

// The palette is final: the reference's host handling of it and the remap of d_in's n pixels (queued, not waited for).
// through_table: the unique list of the quantize (d_uniq / d_cb->ucount, mapped through d_map) holds every colour of d_in.
void remap_quantized(dq_context *ctx, uint32_t n, const uint32_t *d_in, uint32_t *d_out, uint32_t *k_inout, uint32_t *colortable,
                     bool through_table) {
  uint32_t k = dedup_palette(colortable, *k_inout);
  *k_inout = k;
  ctx->stats.actual_colors = k;
  if (n == 0) return;  // (a row shard without rows)
  const uint32_t U = ctx->stats.num_points;
  if (through_table && k <= 256) {
    // the tables ride in the kernel's parameter block: no upload
    MapTablesParam tables;
    int lut[kLutEntries];
    build_search_tables(colortable, (int)k, tables.sorted, lut);
    for (int i = 0; i < kLutEntries; ++i) tables.lut[i] = (uint16_t)lut[i];
    ctx->mark(4);
    map_unique_params(tables, ctx->d_uniq.ptr, &ctx->d_cb->ucount, U, ctx->d_map, (int)k, ctx->sm_count, ctx->stream);
    ctx->mark(5);
    map_gather(d_in, n, d_out, ctx->d_map, ctx->sm_count, ctx->stream);
    ctx->mark(6);
    ctx->mark(7);
    ctx->stats.kernel_launches += 2;
    ctx->stats.remap_path = 2;
  } else if (through_table) {
    upload_search_tables(ctx, colortable, (int)k);
    remap_through_table(ctx, d_in, n, d_out, (int)k, U);
  } else {
    upload_search_tables(ctx, colortable, (int)k);
    remap_bruteforce(ctx, d_in, n, d_out, (int)k);
  }
}

// quant_recurse's remap: through the table when there are at most half as many unique colours as pixels.
void recurse_remap_tail(dq_context *ctx, uint32_t n, const uint32_t *d_in, uint32_t *d_out, uint32_t *k_inout, uint32_t *colortable) {
  const bool through_table = ctx->qs.table_dirty && (uint64_t)ctx->stats.num_points * 2 <= n;
  remap_quantized(ctx, n, d_in, d_out, k_inout, colortable, through_table);
}

void recurse_remap(dq_context *ctx, uint32_t n, const uint32_t *d_in, uint32_t *d_out, uint32_t *k_inout, uint32_t *colortable,
                   std::chrono::steady_clock::time_point *t_palette = nullptr) {
  quantize_finish(ctx, k_inout, colortable);
  if (t_palette) *t_palette = std::chrono::steady_clock::now();
  recurse_remap_tail(ctx, n, d_in, d_out, k_inout, colortable);
}

void quant_recurse_device_impl(dq_context *ctx, uint32_t n, const uint32_t *d_in, uint32_t *d_out, uint32_t *k_inout,
                               uint32_t *colortable, int all_unique, double *ms_quant, double *ms_map) {
  auto t0 = std::chrono::steady_clock::now();
  recurse_begin(ctx, n, d_in, *k_inout, all_unique);
  auto t1 = t0;
  recurse_remap(ctx, n, d_in, d_out, k_inout, colortable, &t1);  // waits for the palette, then queues the remap
  ctx->wait();
  if (ctx->profiling) {
    auto span = [&](int a, int b) {
      float ms = 0.f;
      DQ_CUDA_CHECK(cudaEventElapsedTime(&ms, ctx->ev[a], ctx->ev[b]));
      return ms;
    };
    ctx->stats.stage_ms[0] = span(0, 1);
    ctx->stats.stage_ms[1] = span(1, 2);
    ctx->stats.stage_ms[2] = span(2, 3);
    ctx->stats.stage_ms[3] = span(4, 5);
    ctx->stats.stage_ms[4] = span(5, 6);
    ctx->stats.stage_ms[5] = span(6, 7);
    ctx->stats.stage_ms[6] = span(0, 7);
  }
  auto t2 = std::chrono::steady_clock::now();
  if (ms_quant) *ms_quant = std::chrono::duration<double, std::milli>(t1 - t0).count();
  if (ms_map) *ms_map = std::chrono::duration<double, std::milli>(t2 - t1).count();
}

// ---- quant_recurse over a batch of items (kernels: dq_batch.cu) -------------------------------------------------------
// Fatal like every other bad argument: offsets that decrease or end beyond the input.
void check_batch_offsets(uint32_t num_items, const uint32_t *offsets, uint32_t num_pixels) {
  for (uint32_t i = 0; i < num_items; ++i) {
    if (offsets[i + 1] < offsets[i]) {
      fprintf(stderr, "divquant_b200: batch offsets decrease at item %u (%u -> %u)\n", i, offsets[i], offsets[i + 1]);
      abort();
    }
  }
  if (offsets[num_items] > num_pixels) {
    fprintf(stderr, "divquant_b200: batch offsets end at %u, beyond the %u input pixels\n", offsets[num_items], num_pixels);
    abort();
  }
}

// ... and for quant_recurse, an item with no pixels or K = 0.
void check_batch_args(uint32_t num_items, const uint32_t *offsets, uint32_t num_pixels, const uint32_t *ks) {
  check_batch_offsets(num_items, offsets, num_pixels);
  for (uint32_t i = 0; i < num_items; ++i) check_quant_args(offsets[i + 1] - offsets[i], ks[i], 8);
}

// The batch remap (batch_remap_kernel) of the items added to it: per item its sorted palette, lut_init and, for a label
// image, its label table, plus its pixels cut into kBatchTilePixels tiles.  run() sends all of it up in one copy and
// launches one kernel.
struct BatchRemap {
  std::vector<BatchTile> tiles;
  std::vector<uint2> tabs;  // (offset in sorted, palette size) per item
  std::vector<uint32_t> sorted;
  std::vector<uint16_t> luts, labels;  // labels: one per sorted entry, at the same offsets as sorted

  // pixels [begin, begin + n) of the launch's input mapped to colortable[0, k), k <= kIntColors
  void add(const uint32_t *colortable, uint32_t k, uint32_t begin, uint32_t n, bool with_labels) {
    const uint32_t t = (uint32_t)tabs.size(), off = (uint32_t)sorted.size();
    tabs.push_back(make_uint2(off, k));
    sorted.resize(off + k);
    int lut[kLutEntries];
    build_search_tables(colortable, (int)k, sorted.data() + off, lut);
    for (int e = 0; e < kLutEntries; ++e) luts.push_back((uint16_t)lut[e]);
    if (with_labels) {
      uint32_t lab[kIntColors];
      build_label_table(colortable, (int)k, sorted.data() + off, lab);
      labels.insert(labels.end(), lab, lab + k);
    }
    for (uint32_t b = 0; b < n; b += (uint32_t)kBatchTilePixels)
      tiles.push_back({begin + b, begin + std::min<uint32_t>(n, b + (uint32_t)kBatchTilePixels), t, 0u});
  }

  // d_labels: nullptr, or (when every item was added with labels) the label image.  Returns the kernels launched.
  uint32_t run(dq_context *ctx, const uint32_t *d_in, uint32_t *d_out, uint32_t *d_labels) {
    if (tiles.empty()) return 0;
    // tiles, (offset, size) per item, sorted palettes, lut_init and label tables go up in one copy
    static_assert(sizeof(BatchTile) == 4 * sizeof(uint32_t), "four words per tile");
    const size_t w_tiles = 4 * tiles.size(), w_tabs = 2 * tabs.size(), w_u16 = (luts.size() + labels.size() + 1) / 2;
    const size_t words = w_tiles + w_tabs + sorted.size() + w_u16;
    ctx->b_tab.ensure(words);
    uint32_t *h = ctx->b_tab.ptr;
    memcpy(h, tiles.data(), w_tiles * sizeof(uint32_t));
    memcpy(h + w_tiles, tabs.data(), w_tabs * sizeof(uint32_t));
    memcpy(h + w_tiles + w_tabs, sorted.data(), sorted.size() * sizeof(uint32_t));
    uint16_t *h16 = reinterpret_cast<uint16_t *>(h + w_tiles + w_tabs + sorted.size());
    memcpy(h16, luts.data(), luts.size() * sizeof(uint16_t));
    memcpy(h16 + luts.size(), labels.data(), labels.size() * sizeof(uint16_t));
    ctx->b_tables.ensure(words);
    uint32_t *d = ctx->b_tables.ptr;
    DQ_CUDA_CHECK(cudaMemcpyAsync(d, h, words * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    const uint16_t *d16 = reinterpret_cast<const uint16_t *>(d + w_tiles + w_tabs + sorted.size());
    batch_remap_launch(d_in, d_out, reinterpret_cast<const BatchTile *>(d), (uint32_t)tiles.size(), d + w_tiles + w_tabs,
                       reinterpret_cast<const uint2 *>(d + w_tiles), d16, d16 + luts.size(), d_labels, ctx->stream);
    ctx->wait();
    return 1;
  }
};

// Every item gets what quant_recurse_device_impl gives it alone on this context.  An item is batched when the single call
// would split it on the ordered path in shared memory: weighted (all_unique = 0), K <= kSplit2MaxColors and at most
// min(exact_max_points, kBatchMaxPoints) distinct colours with the ordered path on.  The histogram kernel finds U; any
// other item goes through quant_recurse_device_impl, in item order between the batched items' palette handling, so that
// the "# empty clusters" lines come out as a loop of single calls prints them.  d_labels (optional): every item's
// dq_colortable_indexes (asGreyscale = 0) of its output in its deduped palette, the label image.
void quant_recurse_batch_impl(dq_context *ctx, uint32_t num_items, const uint32_t *offsets, const uint32_t *d_in, uint32_t *d_out,
                              uint32_t *ks, uint32_t *colortables, int all_unique, uint32_t *d_labels) {
  dq_batch_stats &bs = ctx->batch_stats;
  bs = dq_batch_stats();
  bs.items = num_items;
  uint32_t launches = 0;
  const uint32_t base = offsets[0], total = offsets[num_items] - base;
  const uint32_t limit = ctx->exact_small ? std::min<uint32_t>(ctx->exact_max_points, kBatchMaxPoints) : 0u;
  std::vector<uint32_t> cand_of(num_items, UINT32_MAX), cand_pal;
  size_t sum_k = 0;
  for (uint32_t i = 0; i < num_items; ++i) {
    if (all_unique || limit == 0u || ks[i] > kSplit2MaxColors) continue;
    cand_of[i] = (uint32_t)cand_pal.size();
    cand_pal.push_back((uint32_t)sum_k);
    sum_k += ks[i];
  }
  const uint32_t nc = (uint32_t)cand_pal.size();
  const size_t w_items = (size_t)4 * nc, w_res = (size_t)kBatchResultWords * nc;
  if (nc > 0) {
    static_assert(sizeof(BatchItem) == 4 * sizeof(uint32_t), "four words per item");
    ctx->b_work.ensure(w_items + w_res + sum_k + (size_t)3 * total);
    ctx->b_cluster_size.ensure(sum_k);
    ctx->b_cluster_mean.ensure(3 * sum_k);
    ctx->b_up.ensure(w_items);
    BatchItem *h_items = reinterpret_cast<BatchItem *>(ctx->b_up.ptr);
    for (uint32_t i = 0; i < num_items; ++i) {
      const uint32_t j = cand_of[i];
      if (j != UINT32_MAX) h_items[j] = {offsets[i] - base, offsets[i + 1] - offsets[i], ks[i], cand_pal[j]};
    }
    uint32_t *const d_items = ctx->b_work.ptr, *const d_res = d_items + w_items, *const d_pal = d_res + w_res;
    uint32_t *const d_colours = d_pal + sum_k, *const d_counts = d_colours + total, *const d_first = d_counts + total;
    const BatchItem *d_items_b = reinterpret_cast<const BatchItem *>(d_items);
    DQ_CUDA_CHECK(cudaMemcpyAsync(d_items, h_items, w_items * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    batch_hist_launch(d_in + base, d_items_b, nc, d_colours, d_counts, d_first, d_res, ctx->stream);
    batch_split_launch(d_items_b, nc, limit, d_colours, d_counts, d_first, d_res, d_pal, ctx->b_cluster_size.ptr, ctx->b_cluster_mean.ptr,
                       ctx->stream);
    launches += 2;
    // results and palettes of all items come back in one copy
    ctx->b_down.ensure(w_res + sum_k);
    DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->b_down.ptr, d_res, (w_res + sum_k) * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    ctx->wait();
  }
  BatchRemap remap;
  remap.tabs.reserve(nc);
  remap.luts.reserve((size_t)nc * kLutEntries);
  double host_ms = 0.0;
  size_t pal_off = 0;
  for (uint32_t i = 0; i < num_items; ++i) {
    const uint32_t n = offsets[i + 1] - offsets[i];
    uint32_t *const ct = colortables + pal_off;
    pal_off += ks[i];
    const uint32_t j = cand_of[i];
    const uint32_t *r = (j != UINT32_MAX) ? ctx->b_down.ptr + (size_t)kBatchResultWords * j : nullptr;
    if (r != nullptr && r[0] <= limit) {
      const auto t0 = std::chrono::steady_clock::now();
      const uint32_t *ctl = r + 4;
      if (ctl[kCtlError] != 0) {
        fprintf(stderr, "divquant_b200: split of batch item %u failed (code %u; internal error)\n", i, ctl[kCtlError]);
        abort();
      }
      const uint32_t actual = r[1], empty = r[2];
      memcpy(ct, ctx->b_down.ptr + w_res + cand_pal[j], actual * sizeof(uint32_t));
      if (empty) fprintf(stderr, "# empty clusters: %d\n", (int)empty);  // (:1067-1070)
      const uint32_t k = dedup_palette(ct, actual);
      ks[i] = k;
      remap.add(ct, k, offsets[i] - base, n, d_labels != nullptr);
      bs.batched_items++;
      bs.empty_clusters += empty;
      host_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    } else {
      memset(&ctx->stats, 0, sizeof(ctx->stats));
      ctx->stats.num_pixels = n;
      quant_recurse_device_impl(ctx, n, d_in + offsets[i], d_out + offsets[i], &ks[i], ct, all_unique, nullptr, nullptr);
      launches += ctx->stats.kernel_launches;
      bs.empty_clusters += ctx->stats.empty_clusters;
      bs.single_call_items++;
      if (d_labels != nullptr) {
        dq_colortable_indexes_device(ctx, d_out + offsets[i], n, ct, (int)ks[i], d_labels + offsets[i], 0);
        launches++;  // map_labels
      }
    }
  }
  launches += remap.run(ctx, d_in + base, d_out + base, d_labels != nullptr ? d_labels + base : nullptr);
  memset(&ctx->stats, 0, sizeof(ctx->stats));  // (dq_call_stats describes one frame: only the launches are kept)
  ctx->stats.kernel_launches = launches;
  bs.kernel_launches = launches;
  bs.host_palette_ms = (float)host_ms;
}

// Fatal before any device work: bad offsets, an empty palette, and with labels a palette above dq_colortable_indexes'
// limit.
void check_map_batch_args(uint32_t num_items, const uint32_t *offsets, uint32_t num_pixels, const int *sizes, bool labels) {
  check_batch_offsets(num_items, offsets, num_pixels);
  for (uint32_t i = 0; i < num_items; ++i) {
    if (sizes[i] <= 0) {
      fprintf(stderr, "divquant_b200: batch item %u has a colortable of %d entries; map_colors_mps needs a non-empty one\n", i,
              sizes[i]);
      abort();  // assert(num_colors > 0) (:266)
    }
    if (labels && sizes[i] > 24000) {
      fprintf(stderr, "divquant_b200: batch item %u has a colortable of %d entries; label images support 1..24000\n", i, sizes[i]);
      abort();
    }
  }
}

// Every item gets what dq_map_colors_device (prefer_table = 1) gives it alone on this context, and with d_labels its
// dq_colortable_indexes (asGreyscale = 0).  Items whose palette fits the integer arg-min (<= kIntColors entries) go
// through one batch remap launch; the others run the single call in item order.  Items with no pixels write nothing.
void map_colors_batch_impl(dq_context *ctx, uint32_t num_items, const uint32_t *offsets, const uint32_t *d_in, uint32_t *d_out,
                           const int *sizes, const uint32_t *colortables, uint32_t *d_labels) {
  dq_batch_stats &bs = ctx->batch_stats;
  bs = dq_batch_stats();
  bs.items = num_items;
  uint32_t launches = 0;
  const uint32_t base = offsets[0];
  BatchRemap remap;
  double host_ms = 0.0;
  size_t pal_off = 0;
  for (uint32_t i = 0; i < num_items; ++i) {
    const uint32_t n = offsets[i + 1] - offsets[i];
    const int k = sizes[i];
    const uint32_t *const ct = colortables + pal_off;
    pal_off += (size_t)k;
    if (k <= kIntColors) {
      bs.batched_items++;
      if (n == 0) continue;
      const auto t0 = std::chrono::steady_clock::now();
      remap.add(ct, (uint32_t)k, offsets[i] - base, n, d_labels != nullptr);
      host_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    } else {
      bs.single_call_items++;
      if (n == 0) continue;
      dq_map_colors_device(ctx, d_in + offsets[i], n, d_out + offsets[i], ct, k, 1);
      launches += ctx->stats.kernel_launches;
      if (d_labels != nullptr) {
        dq_colortable_indexes_device(ctx, d_out + offsets[i], n, ct, k, d_labels + offsets[i], 0);
        launches++;  // map_labels
      }
    }
  }
  launches += remap.run(ctx, d_in + base, d_out + base, d_labels != nullptr ? d_labels + base : nullptr);
  memset(&ctx->stats, 0, sizeof(ctx->stats));  // (as after a quant_recurse batch: only the launches are kept)
  ctx->stats.kernel_launches = launches;
  bs.kernel_launches = launches;
  bs.host_palette_ms = (float)host_ms;
}

// ---- every region of a tag image in one call (kernels: dq_regions.cu) ------------------------------------------------
// Fatal before any device work: more than 2^24 regions (the sort's three digit passes).
void check_region_count(uint32_t num_regions, const char *call) {
  if (num_regions > (1u << 24)) {
    fprintf(stderr, "divquant_b200: %u regions; %s takes at most 2^24\n", num_regions, call);
    abort();
  }
}

// ... and for quant_recurse, a region asking for K = 0.
void check_regions_args(uint32_t num_regions, const uint32_t *ks) {
  check_region_count(num_regions, "dq_quant_regions");
  for (uint32_t r = 0; r < num_regions; ++r) {
    if (ks[r] == 0) {
      fprintf(stderr, "divquant_b200: region %u requests K = 0\n", r);
      abort();  // assert(num_colors > 0) (:266)
    }
  }
}

// ... and for map_colors_mps, a palette of negative size and, with labels, one above dq_colortable_indexes' limit.
void check_map_regions_args(uint32_t num_regions, const int *sizes, bool labels) {
  check_region_count(num_regions, "dq_map_regions");
  for (uint32_t r = 0; r < num_regions; ++r) {
    if (sizes[r] < 0) {
      fprintf(stderr, "divquant_b200: region %u has a colortable of %d entries\n", r, sizes[r]);
      abort();
    }
    if (labels && sizes[r] > 24000) {
      fprintf(stderr, "divquant_b200: region %u has a colortable of %d entries; label images support 1..24000\n", r, sizes[r]);
      abort();
    }
  }
}

// The pixels of a tag image partitioned by region on the device (dq_regions.cu), which both regions calls work on.
struct RegionPartition {
  const uint32_t *off = nullptr;  // HOST, num_regions + 1: region r = sorted positions [off[r], off[r + 1]), off[num_regions] = m
  uint32_t m = 0, launches = 0;
  const uint2 *sorted = nullptr;  // the m (tag, index) pairs in region order
  uint32_t *g_in = nullptr, *g_out = nullptr, *g_labels = nullptr;  // in, out and labels in that order (g_labels: with labels)
};

// h_dropped: nullptr, or a host bitmap of (num_regions + 31) / 32 words; the pixels of the regions set in it are left out
// like pixels in no region, so those regions come back with no pixels.
RegionPartition partition_regions(dq_context *ctx, uint32_t n, const uint32_t *d_in, const uint32_t *d_tags, uint32_t num_regions,
                                  const uint32_t *h_dropped, bool labels) {
  RegionPartition rp;
  ctx->r_offsets.ensure((size_t)num_regions + 1);
  uint32_t *const off = ctx->r_offsets.ptr;
  rp.off = off;
  if (n == 0) {
    memset(off, 0, ((size_t)num_regions + 1) * sizeof(uint32_t));
    return rp;
  }
  const size_t scratch = region_scratch_words(n, num_regions), dropped_words = h_dropped != nullptr ? ((size_t)num_regions + 31) / 32 : 0;
  ctx->r_pairs.ensure(2 * (size_t)n);
  ctx->r_px.ensure((labels ? 3 : 2) * (size_t)n);
  ctx->r_scratch.ensure(scratch + dropped_words);
  uint32_t *const d_dropped = h_dropped != nullptr ? ctx->r_scratch.ptr + scratch : nullptr;
  if (d_dropped != nullptr)
    DQ_CUDA_CHECK(cudaMemcpyAsync(d_dropped, h_dropped, dropped_words * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  rp.g_in = ctx->r_px.ptr;
  rp.g_out = rp.g_in + n;
  rp.g_labels = labels ? rp.g_out + n : nullptr;
  rp.launches = region_partition(d_in, d_tags, n, num_regions, d_dropped, ctx->r_pairs.ptr, rp.g_in, ctx->r_scratch.ptr, &rp.sorted,
                                 ctx->stream);
  DQ_CUDA_CHECK(cudaMemcpyAsync(off, region_offsets(ctx->r_scratch.ptr, n), ((size_t)num_regions + 1) * sizeof(uint32_t),
                                cudaMemcpyDeviceToHost, ctx->stream));
  ctx->wait();
  rp.m = off[num_regions];
  return rp;
}

// The gathered out (and labels) back to image layout at the partitioned pixels, and the call's statistics.
void finish_regions(dq_context *ctx, const RegionPartition &rp, uint32_t num_regions, uint32_t launches, uint32_t *d_out,
                    uint32_t *d_labels) {
  if (rp.m > 0) {
    region_scatter_back(rp.sorted, rp.m, rp.g_out, rp.g_labels, d_out, d_labels, ctx->stream);
    launches++;
    ctx->wait();
  }
  dq_batch_stats &bs = ctx->batch_stats;
  bs.items = num_regions;
  bs.kernel_launches = launches;
  memset(&ctx->stats, 0, sizeof(ctx->stats));  // (as after a batch: only the launches are kept)
  ctx->stats.kernel_launches = launches;
}

// quant_recurse_batch_impl over the regions of a tag image: the pixels partitioned by tag, the regions with pixels
// quantized as the batch's items in region order, the results scattered back to image layout.
void quant_regions_impl(dq_context *ctx, uint32_t n, const uint32_t *d_in, const uint32_t *d_tags, uint32_t num_regions,
                        uint32_t *d_out, uint32_t *ks, uint32_t *colortables, uint32_t *d_labels) {
  const RegionPartition rp = partition_regions(ctx, n, d_in, d_tags, num_regions, nullptr, d_labels != nullptr);
  const uint32_t *const off = rp.off;
  uint32_t launches = rp.launches;
  // the regions with pixels, in region order, are the batch's items; their palettes are packed by requested K
  std::vector<uint32_t> item_off, item_k, item_region;
  size_t item_pal = 0;
  for (uint32_t r = 0; r < num_regions; ++r) {
    if (off[r + 1] == off[r]) continue;
    item_off.push_back(off[r]);
    item_k.push_back(ks[r]);
    item_region.push_back(r);
    item_pal += ks[r];
  }
  item_off.push_back(rp.m);
  const uint32_t num_items = (uint32_t)item_region.size();
  std::vector<uint32_t> pal(std::max<size_t>(item_pal, 1));
  if (num_items > 0) {
    quant_recurse_batch_impl(ctx, num_items, item_off.data(), rp.g_in, rp.g_out, item_k.data(), pal.data(), 0, rp.g_labels);
    launches += ctx->batch_stats.kernel_launches;
  } else {
    ctx->batch_stats = dq_batch_stats();
  }
  // palettes and actual K into the caller's packing (requested K of every region, the empty ones included)
  size_t at = 0, from = 0;
  for (uint32_t r = 0, i = 0; r < num_regions; ++r) {
    const uint32_t requested = ks[r];
    if (i < num_items && item_region[i] == r) {
      memcpy(colortables + at, pal.data() + from, item_k[i] * sizeof(uint32_t));
      from += requested;
      ks[r] = item_k[i++];
    } else {
      ks[r] = 0;
    }
    at += requested;
  }
  finish_regions(ctx, rp, num_regions, launches, d_out, d_labels);
}

// map_colors_batch_impl over the regions of a tag image: the pixels partitioned by tag, the mapped regions with pixels
// remapped as the batch's items in region order, the results scattered back to image layout.  A region with an empty
// palette is not mapped: the partition drops its pixels as it drops those in no region, so they are never sorted,
// gathered or scattered.
void map_regions_impl(dq_context *ctx, uint32_t n, const uint32_t *d_in, const uint32_t *d_tags, uint32_t num_regions,
                      const int *sizes, const uint32_t *colortables, uint32_t *d_out, uint32_t *d_labels) {
  std::vector<uint32_t> dropped;  // only when some region is unmapped
  for (uint32_t r = 0; r < num_regions; ++r) {
    if (sizes[r] != 0) continue;
    if (dropped.empty()) dropped.assign(((size_t)num_regions + 31) / 32, 0u);
    dropped[r >> 5] |= 1u << (r & 31u);
  }
  const RegionPartition rp = partition_regions(ctx, n, d_in, d_tags, num_regions, dropped.empty() ? nullptr : dropped.data(),
                                               d_labels != nullptr);
  const uint32_t *const off = rp.off;
  uint32_t launches = rp.launches;
  // the regions with pixels, in region order, are the batch's items, with their palettes packed end to end
  std::vector<uint32_t> item_off, packed;
  std::vector<int> item_size;
  size_t at = 0;
  for (uint32_t r = 0; r < num_regions; ++r) {
    const uint32_t *const ct = colortables + at;
    at += (size_t)sizes[r];
    if (off[r + 1] == off[r]) continue;
    item_off.push_back(off[r]);
    item_size.push_back(sizes[r]);
    packed.insert(packed.end(), ct, ct + sizes[r]);
  }
  item_off.push_back(rp.m);
  const uint32_t num_items = (uint32_t)item_size.size();
  if (num_items > 0) {
    map_colors_batch_impl(ctx, num_items, item_off.data(), rp.g_in, rp.g_out, item_size.data(), packed.data(), rp.g_labels);
    launches += ctx->batch_stats.kernel_launches;
  } else {
    ctx->batch_stats = dq_batch_stats();
  }
  finish_regions(ctx, rp, num_regions, launches, d_out, d_labels);
}

std::mutex g_default_mutex;
dq_context *g_default = nullptr;
// The reference's functions are re-entrant; the entry points that run on the one lazily created default context are
// serialised instead: each holds this lock for the whole call (recursive: dq_quant_blocks calls other entry points).
std::recursive_mutex g_default_call_mutex;
struct DefaultLock {
  std::lock_guard<std::recursive_mutex> guard;
  DefaultLock() : guard(g_default_call_mutex) {}
};
int g_display_timings = -1;

int display_timings_default() {
  if (g_display_timings < 0) {
    const char *e = getenv("DIVQUANT_B200_TIMINGS");
    g_display_timings = (e && e[0] == '0') ? 0 : 1;
  }
  return g_display_timings;
}

}  // namespace

// =====================================================================================================
// extern "C" layer
// =====================================================================================================
extern "C" {

const char *dq_version(void) { return "divquant_b200 0.1 (sm_100a)"; }

uint32_t dq_host_dedup_palette(uint32_t *colortable, uint32_t num_colors) { return dedup_palette(colortable, num_colors); }

void dq_host_build_search_tables(const uint32_t *colortable, int num_colors, uint32_t *sorted_out, int32_t *lut_init_out) {
  build_search_tables(colortable, num_colors, sorted_out, lut_init_out);
}

void dq_host_build_label_table(const uint32_t *colortable, int num_colors, uint32_t *labels_out) {
  std::vector<uint32_t> sorted((size_t)num_colors);
  int lut[kLutEntries];
  build_search_tables(colortable, num_colors, sorted.data(), lut);
  build_label_table(colortable, num_colors, sorted.data(), labels_out);
}

uint32_t dq_host_select_cut_overrides(const uint32_t *begin, const uint32_t *size, const uint32_t *status, uint32_t n,
                                      uint32_t already, uint32_t *picked_out) {
  if (n > kTieListCap) n = kTieListCap;
  CutOverride rec[kTieListCap], out[kCutOverrideCap];
  for (uint32_t i = 0; i < n; ++i) rec[i].begin = begin[i], rec[i].size = size[i], rec[i].mean_here = (double)i, rec[i].mean_ref = 0.0;
  uint32_t n_out = std::min(already, kCutOverrideCap);
  const uint32_t first = n_out;
  const uint32_t added = select_cut_overrides(rec, status, n, out, &n_out, kCutOverrideCap);
  for (uint32_t k = 0; k < added; ++k) picked_out[k] = (uint32_t)out[first + k].mean_here;  // the entry's index
  return added;
}

dq_context *dq_context_create(int device) {
  int count = 0;
  cudaError_t err = cudaGetDeviceCount(&count);
  if (err != cudaSuccess || count == 0) {
    fprintf(stderr, "divquant_b200: no CUDA device available (%s); this library has no CPU fallback\n",
            err != cudaSuccess ? cudaGetErrorString(err) : "device count is 0");
    abort();
  }
  dq_context *ctx = new dq_context();
  if (device < 0) DQ_CUDA_CHECK(cudaGetDevice(&device));
  ctx->device = device;
  DQ_CUDA_CHECK(cudaSetDevice(device));
  cudaDeviceProp prop;
  DQ_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    fprintf(stderr, "divquant_b200: device %d (%s, sm_%d%d) is not a Blackwell sm_100a part\n", device, prop.name,
            prop.major, prop.minor);
    abort();
  }
  ctx->sm_count = prop.multiProcessorCount;
  ctx->split_ctas = 0;  // 0 = as many as can be co-resident
  if (const char *e = getenv("DIVQUANT_B200_SPLIT_CTAS")) ctx->split_ctas = std::max(atoi(e), 0);
  DQ_CUDA_CHECK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  DQ_CUDA_CHECK(cudaMalloc(&ctx->d_table, (size_t)kColourBins * sizeof(uint32_t)));
  DQ_CUDA_CHECK(cudaMemsetAsync(ctx->d_table, 0, (size_t)kColourBins * sizeof(uint32_t), ctx->stream));
  DQ_CUDA_CHECK(cudaMalloc(&ctx->d_map, (size_t)kColourBins * sizeof(uint32_t)));
  DQ_CUDA_CHECK(cudaMalloc(&ctx->d_cb, sizeof(ControlBlock)));
  DQ_CUDA_CHECK(cudaMallocHost(&ctx->h_cb, sizeof(ControlBlock)));
  {
    void *mb = nullptr;
    DQ_CUDA_CHECK(cudaHostAlloc(&mb, kMailboxWords * sizeof(uint32_t), cudaHostAllocMapped));
    memset(mb, 0, kMailboxWords * sizeof(uint32_t));
    ctx->mailbox = static_cast<volatile uint32_t *>(mb);
  }
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  for (int i = 0; i < 8; ++i) DQ_CUDA_CHECK(cudaEventCreate(&ctx->ev[i]));
  ctx->display_timings = display_timings_default();
  if (const char *e = getenv("DIVQUANT_B200_TIE")) ctx->tie_policy = std::min(std::max(atoi(e), 0), 2);
  if (const char *e = getenv("DIVQUANT_B200_RESOLVE")) ctx->resolve_mode = atoi(e) & 3;
  if (const char *e = getenv("DIVQUANT_B200_SPIN_MS")) ctx->spin_cycles = (long long)std::max(atol(e), 0l) * 2000000ll;  // ~2 GHz
  if (const char *e = getenv("DIVQUANT_B200_EXACT_SMALL")) ctx->exact_small = (e[0] != '0');
  if (const char *e = getenv("DIVQUANT_B200_EXACT_MAX")) ctx->exact_max_points = (uint32_t)std::min<long>(std::max<long>(atol(e), 0), kExactMaxPoints);
  ctx->profile_narrow = getenv("DQ_PROFILE_NARROW") != nullptr;
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  return ctx;
}

void dq_context_set_split_ctas(dq_context *ctx, int num_ctas) {
  require_device(ctx);
  ctx->split_ctas = num_ctas >= 1 ? num_ctas : 0;  // clamped to the co-residency limit at launch
}

void dq_context_set_exact_small(dq_context *ctx, int enabled) { ctx->exact_small = enabled ? 1 : 0; }
void dq_context_set_tie_policy(dq_context *ctx, int policy) { ctx->tie_policy = std::min(std::max(policy, 0), 2); }
void dq_context_set_exact_max_points(dq_context *ctx, uint32_t max_points) {
  ctx->exact_max_points = std::min<uint32_t>(max_points, kExactMaxPoints);
}

void dq_context_destroy(dq_context *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  ctx->d_in.release();
  ctx->d_out.release();
  ctx->d_uniq.release();
  ctx->d_pts0.release();
  ctx->d_pts1.release();
  ctx->d_keys.release();
  ctx->d_nodes.release();
  ctx->d_jobs.release();
  ctx->d_acc.release();
  ctx->d_ctl_i32.release();
  ctx->d_ctl_f64.release();
  ctx->d_palette.release();
  ctx->d_cluster_size.release();
  ctx->d_sorted.release();
  ctx->d_cluster_mean.release();
  ctx->d_records.release();
  ctx->d_pal_scratch.release();
  ctx->d_timeline.release();
  ctx->d_slots.release();
  ctx->d_progress.release();
  ctx->d_exact.release();
  ctx->d_tie.release();
  ctx->d_ovr.release();
  ctx->d_flat.release();
  ctx->d_sortvals.release();
  ctx->b_work.release();
  ctx->b_tables.release();
  ctx->b_labels.release();
  ctx->b_cluster_size.release();
  ctx->b_cluster_mean.release();
  ctx->b_up.release();
  ctx->b_down.release();
  ctx->b_tab.release();
  ctx->r_pairs.release();
  ctx->r_px.release();
  ctx->r_scratch.release();
  ctx->r_offsets.release();
  cudaFree(ctx->d_table);
  cudaFree(ctx->d_map);
  cudaFree(ctx->d_cb);
  cudaFreeHost(ctx->h_cb);
  if (ctx->h_small) cudaFreeHost(ctx->h_small);
  if (ctx->mailbox) cudaFreeHost(const_cast<uint32_t *>(ctx->mailbox));
  for (int i = 0; i < 8; ++i) cudaEventDestroy(ctx->ev[i]);
  if (ctx->wait_ev) cudaEventDestroy(ctx->wait_ev);
  if (ctx->tie_ev) cudaEventDestroy(ctx->tie_ev);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

dq_context *dq_default_context(void) {
  std::lock_guard<std::mutex> lock(g_default_mutex);
  if (!g_default) g_default = dq_context_create(-1);
  return g_default;
}

void *dq_context_stream(dq_context *ctx) { return (void *)ctx->stream; }

void dq_context_synchronize(dq_context *ctx) {
  require_device(ctx);
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}

void dq_context_last_stats(const dq_context *ctx, dq_call_stats *out) { *out = ctx->stats; }

void dq_context_set_profiling(dq_context *ctx, int enabled) { ctx->profiling = enabled ? 1 : 0; }

void dq_set_display_timings(int enabled) {
  g_display_timings = enabled ? 1 : 0;
  std::lock_guard<std::mutex> lock(g_default_mutex);
  if (g_default) g_default->display_timings = g_display_timings;
}

int dq_validate_num_bits(unsigned char num_bits) {
  if (!(0 < num_bits && num_bits <= 8)) {
    fprintf(stderr, "Number of bits per channel ( %d ) must be in [1,8] !\n", num_bits);
    return 0;
  }
  return 1;
}

double dq_get_double_scale(const uint32_t * /*inPixels*/, uint32_t numPixels) { return sample_norm(1, numPixels, 1); }

// ---- device-pointer entry points ----

void dq_quant_recurse_device(dq_context *ctx, uint32_t numPixels, const uint32_t *d_in, uint32_t *d_out,
                             uint32_t *numClustersPtr, uint32_t *outColortablePtr, int allPixelsUnique) {
  require_device(ctx);
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  ctx->stats.num_pixels = numPixels;
  quant_recurse_device_impl(ctx, numPixels, d_in, d_out, numClustersPtr, outColortablePtr, allPixelsUnique, nullptr, nullptr);
}

void dq_quant_varpart_device(dq_context *ctx, uint32_t numPixels, const uint32_t *d_in, uint32_t numRows, uint32_t numCols,
                             uint32_t *numClustersPtr, uint32_t *colortablePtr, int num_bits, int dec_factor, int max_iters,
                             int allPixelsUnique) {
  require_device(ctx);
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  ctx->stats.num_pixels = numPixels;
  const bool dirty = quantize_device(ctx, numPixels, d_in, numRows, numCols, numClustersPtr, colortablePtr, num_bits,
                                     dec_factor, max_iters, allPixelsUnique, nullptr, nullptr, nullptr);
  (void)dirty;
}

void dq_map_colors_device(dq_context *ctx, const uint32_t *d_in, uint32_t numPixels, uint32_t *d_out,
                          const uint32_t *colortablePtr, int colormapSize, int prefer_table) {
  require_device(ctx);
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  ctx->stats.num_pixels = numPixels;
  if (colormapSize <= 0) {
    fprintf(stderr, "divquant_b200: map_colors_mps needs a non-empty colortable\n");
    abort();  // assert(num_colors > 0) (:266)
  }
  ctx->stats.actual_colors = (uint32_t)colormapSize;
  upload_search_tables(ctx, colortablePtr, colormapSize);
  bool done = false;
  if (prefer_table && numPixels >= (1u << 16)) {
    // A histogram costs about one pass over the pixels; it pays off when few colours repeat often.
    reset_control(ctx);
    run_histogram(ctx, d_in, numPixels, 1, numPixels, 1, 8);
    DQ_CUDA_CHECK(cudaMemcpyAsync(&ctx->h_cb->ucount, &ctx->d_cb->ucount, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    const uint32_t U = ctx->h_cb->ucount;
    ctx->stats.num_points = U;
    if ((uint64_t)U * 4 <= numPixels) {
      remap_through_table(ctx, d_in, numPixels, d_out, colormapSize, U);
      done = true;
    }
    // no hist_collect ran here, so the counters are zeroed explicitly
    table_clear(ctx->d_uniq.ptr, &ctx->d_cb->ucount, U, ctx->d_table, ctx->sm_count, ctx->stream);
    ctx->stats.kernel_launches++;
  }
  if (!done) remap_bruteforce(ctx, d_in, numPixels, d_out, colormapSize);
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}

void dq_quant_recurse_batch_device(dq_context *ctx, uint32_t num_items, const uint32_t *offsets, uint32_t numPixels, const uint32_t *d_in,
                                   uint32_t *d_out, uint32_t *numClusters, uint32_t *colortables, int allPixelsUnique) {
  if (num_items == 0) return;
  require_device(ctx);
  check_batch_args(num_items, offsets, numPixels, numClusters);
  quant_recurse_batch_impl(ctx, num_items, offsets, d_in, d_out, numClusters, colortables, allPixelsUnique, nullptr);
}

void dq_map_colors_batch_device(dq_context *ctx, uint32_t num_items, const uint32_t *offsets, uint32_t numPixels, const uint32_t *d_in,
                                uint32_t *d_out, const int *colormapSizes, const uint32_t *colortables, uint32_t *d_labels) {
  if (num_items == 0) return;
  require_device(ctx);
  check_map_batch_args(num_items, offsets, numPixels, colormapSizes, d_labels != nullptr);
  map_colors_batch_impl(ctx, num_items, offsets, d_in, d_out, colormapSizes, colortables, d_labels);
}

void dq_quant_regions_device(dq_context *ctx, uint32_t numPixels, const uint32_t *d_in, const uint32_t *d_tags, uint32_t num_regions,
                             uint32_t *d_out, uint32_t *ks, uint32_t *colortables, uint32_t *d_labels) {
  if (num_regions == 0) return;
  require_device(ctx);
  check_regions_args(num_regions, ks);
  quant_regions_impl(ctx, numPixels, d_in, d_tags, num_regions, d_out, ks, colortables, d_labels);
}

void dq_map_regions_device(dq_context *ctx, uint32_t numPixels, const uint32_t *d_in, const uint32_t *d_tags, uint32_t num_regions,
                           const int *colormapSizes, const uint32_t *colortables, uint32_t *d_out, uint32_t *d_labels) {
  if (num_regions == 0 || numPixels == 0) return;
  require_device(ctx);
  check_map_regions_args(num_regions, colormapSizes, d_labels != nullptr);
  map_regions_impl(ctx, numPixels, d_in, d_tags, num_regions, colormapSizes, colortables, d_out, d_labels);
}

void dq_context_last_batch_stats(const dq_context *ctx, dq_batch_stats *out) { *out = ctx->batch_stats; }

// ---- host-pointer entry points ----

void dq_quant_recurse_batch_ctx(dq_context *ctx, uint32_t num_items, const uint32_t *offsets, uint32_t numPixels, const uint32_t *inPixels,
                                uint32_t *outPixels, uint32_t *numClusters, uint32_t *colortables, int allPixelsUnique) {
  if (num_items == 0) return;
  require_device(ctx);
  check_batch_args(num_items, offsets, numPixels, numClusters);
  // only the pixels the items cover travel, from offsets[0] on
  const uint32_t base = offsets[0], total = offsets[num_items] - base;
  std::vector<uint32_t> local(offsets, offsets + num_items + 1);
  for (uint32_t &o : local) o -= base;
  ctx->d_in.ensure(total);
  ctx->d_out.ensure(total);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, inPixels + base, (size_t)total * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  quant_recurse_batch_impl(ctx, num_items, local.data(), ctx->d_in.ptr, ctx->d_out.ptr, numClusters, colortables, allPixelsUnique,
                           nullptr);
  DQ_CUDA_CHECK(cudaMemcpyAsync(outPixels + base, ctx->d_out.ptr, (size_t)total * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}

void dq_map_colors_batch_ctx(dq_context *ctx, uint32_t num_items, const uint32_t *offsets, uint32_t numPixels, const uint32_t *inPixels,
                             uint32_t *outPixels, const int *colormapSizes, const uint32_t *colortables, uint32_t *labels) {
  if (num_items == 0) return;
  require_device(ctx);
  check_map_batch_args(num_items, offsets, numPixels, colormapSizes, labels != nullptr);
  // only the pixels the items cover travel, from offsets[0] on
  const uint32_t base = offsets[0], total = offsets[num_items] - base;
  std::vector<uint32_t> local(offsets, offsets + num_items + 1);
  for (uint32_t &o : local) o -= base;
  ctx->d_in.ensure(total);
  ctx->d_out.ensure(total);
  if (labels != nullptr) ctx->b_labels.ensure(total);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, inPixels + base, (size_t)total * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  map_colors_batch_impl(ctx, num_items, local.data(), ctx->d_in.ptr, ctx->d_out.ptr, colormapSizes, colortables,
                        labels != nullptr ? ctx->b_labels.ptr : nullptr);
  DQ_CUDA_CHECK(cudaMemcpyAsync(outPixels + base, ctx->d_out.ptr, (size_t)total * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (labels != nullptr)
    DQ_CUDA_CHECK(cudaMemcpyAsync(labels + base, ctx->b_labels.ptr, (size_t)total * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}

void dq_quant_regions_ctx(dq_context *ctx, uint32_t numPixels, const uint32_t *inPixels, const uint32_t *tags, uint32_t num_regions,
                          uint32_t *outPixels, uint32_t *ks, uint32_t *colortables, uint32_t *labels) {
  if (num_regions == 0) return;
  require_device(ctx);
  check_regions_args(num_regions, ks);
  // d_in = [pixels | tags], d_out = [out | labels]; out and labels go up too, so that pixels in no region keep them
  const size_t n = numPixels, bytes = n * sizeof(uint32_t);
  ctx->d_in.ensure(2 * n);
  ctx->d_out.ensure(2 * n);
  uint32_t *const d_out = ctx->d_out.ptr, *const d_labels = labels != nullptr ? d_out + n : nullptr;
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, inPixels, bytes, cudaMemcpyHostToDevice, ctx->stream));
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr + n, tags, bytes, cudaMemcpyHostToDevice, ctx->stream));
  DQ_CUDA_CHECK(cudaMemcpyAsync(d_out, outPixels, bytes, cudaMemcpyHostToDevice, ctx->stream));
  if (labels != nullptr) DQ_CUDA_CHECK(cudaMemcpyAsync(d_labels, labels, bytes, cudaMemcpyHostToDevice, ctx->stream));
  quant_regions_impl(ctx, numPixels, ctx->d_in.ptr, ctx->d_in.ptr + n, num_regions, d_out, ks, colortables, d_labels);
  DQ_CUDA_CHECK(cudaMemcpyAsync(outPixels, d_out, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (labels != nullptr) DQ_CUDA_CHECK(cudaMemcpyAsync(labels, d_labels, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}

void dq_map_regions_ctx(dq_context *ctx, uint32_t numPixels, const uint32_t *inPixels, const uint32_t *tags, uint32_t num_regions,
                        const int *colormapSizes, const uint32_t *colortables, uint32_t *outPixels, uint32_t *labels) {
  if (num_regions == 0 || numPixels == 0) return;
  require_device(ctx);
  check_map_regions_args(num_regions, colormapSizes, labels != nullptr);
  // as dq_quant_regions_ctx: d_in = [pixels | tags], d_out = [out | labels], out and labels up and down
  const size_t n = numPixels, bytes = n * sizeof(uint32_t);
  ctx->d_in.ensure(2 * n);
  ctx->d_out.ensure(2 * n);
  uint32_t *const d_out = ctx->d_out.ptr, *const d_labels = labels != nullptr ? d_out + n : nullptr;
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, inPixels, bytes, cudaMemcpyHostToDevice, ctx->stream));
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr + n, tags, bytes, cudaMemcpyHostToDevice, ctx->stream));
  DQ_CUDA_CHECK(cudaMemcpyAsync(d_out, outPixels, bytes, cudaMemcpyHostToDevice, ctx->stream));
  if (labels != nullptr) DQ_CUDA_CHECK(cudaMemcpyAsync(d_labels, labels, bytes, cudaMemcpyHostToDevice, ctx->stream));
  map_regions_impl(ctx, numPixels, ctx->d_in.ptr, ctx->d_in.ptr + n, num_regions, colormapSizes, colortables, d_out, d_labels);
  DQ_CUDA_CHECK(cudaMemcpyAsync(outPixels, d_out, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  if (labels != nullptr) DQ_CUDA_CHECK(cudaMemcpyAsync(labels, d_labels, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}


void dq_quant_recurse_ctx(dq_context *ctx, uint32_t numPixels, const uint32_t *inPixelsPtr, uint32_t *outPixelsPtr,
                          uint32_t *numClustersPtr, uint32_t *outColortablePtr, int allPixelsUnique) {
  require_device(ctx);
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  ctx->stats.num_pixels = numPixels;
  check_quant_args(numPixels, *numClustersPtr, 8);
  ctx->d_in.ensure(numPixels);
  ctx->d_out.ensure(numPixels);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, inPixelsPtr, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  double ms_quant = 0, ms_map = 0;
  quant_recurse_device_impl(ctx, numPixels, ctx->d_in.ptr, ctx->d_out.ptr, numClustersPtr, outColortablePtr, allPixelsUnique,
                            &ms_quant, &ms_map);
  auto t0 = std::chrono::steady_clock::now();
  DQ_CUDA_CHECK(cudaMemcpyAsync(outPixelsPtr, ctx->d_out.ptr, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  ms_map += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (ctx->display_timings) {
    // the reference's two stdout lines (quant_util.cpp:62-66, 141-145), wall clock instead of clock()
    printf("quant_varpart_fast() elapsed: %ld ms aka %0.2f s\n", (long)ms_quant, (float)((long)ms_quant / 1000.0f));
    printf("map_colors_mps() elapsed: %ld ms aka %0.2f s\n", (long)ms_map, (float)((long)ms_map / 1000.0f));
  }
}

void dq_quant_recurse(uint32_t numPixels, const uint32_t *inPixelsPtr, uint32_t *outPixelsPtr, uint32_t *numClustersPtr,
                      uint32_t *outColortablePtr, int allPixelsUnique) {
  DefaultLock lock;
  dq_quant_recurse_ctx(dq_default_context(), numPixels, inPixelsPtr, outPixelsPtr, numClustersPtr, outColortablePtr,
                       allPixelsUnique);
}

void dq_quant_varpart_fast(uint32_t numPixels, const uint32_t *inPixels, uint32_t * /*tmpPixels*/, uint32_t numRows,
                           uint32_t numCols, uint32_t *numClustersPtr, uint32_t *colortablePtr, int num_bits, int dec_factor,
                           int max_iters, int allPixelsUnique) {
  dq_context *ctx = dq_default_context();
  DefaultLock lock;
  require_device(ctx);
  ctx->d_in.ensure(numPixels);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, inPixels, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  dq_quant_varpart_device(ctx, numPixels, ctx->d_in.ptr, numRows, numCols, numClustersPtr, colortablePtr, num_bits, dec_factor,
                          max_iters, allPixelsUnique);
}

void dq_map_colors_mps(const uint32_t *inPixelsPtr, uint32_t numPixels, uint32_t *outPixelsPtr, const uint32_t *colortablePtr,
                       int colormapSize) {
  dq_context *ctx = dq_default_context();
  DefaultLock lock;
  require_device(ctx);
  if (numPixels == 0) return;
  ctx->d_in.ensure(numPixels);
  ctx->d_out.ensure(numPixels);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, inPixelsPtr, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  dq_map_colors_device(ctx, ctx->d_in.ptr, numPixels, ctx->d_out.ptr, colortablePtr, colormapSize, 1);
  DQ_CUDA_CHECK(cudaMemcpyAsync(outPixelsPtr, ctx->d_out.ptr, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}

void dq_cut_bits(const uint32_t *inPixels, uint32_t numPixels, uint32_t *outPixels, unsigned char num_bits_red,
                 unsigned char num_bits_green, unsigned char num_bits_blue) {
  if (!dq_validate_num_bits(num_bits_red) || !dq_validate_num_bits(num_bits_green) || !dq_validate_num_bits(num_bits_blue))
    return;  // silent return after the message, like the reference (DivQuantUni.cpp:41-46)
  if (numPixels == 0) return;
  dq_context *ctx = dq_default_context();
  DefaultLock lock;
  require_device(ctx);
  ctx->d_in.ensure(numPixels);
  ctx->d_out.ensure(numPixels);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, inPixels, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  cut_bits_device(ctx->d_in.ptr, numPixels, ctx->d_out.ptr, num_bits_red, num_bits_green, num_bits_blue, ctx->sm_count, ctx->stream);
  DQ_CUDA_CHECK(cudaMemcpyAsync(outPixels, ctx->d_out.ptr, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}

int dq_calc_color_table(const uint32_t *inPixels, uint32_t numPixels, uint32_t *outPixels, uint32_t numRows, uint32_t numCols,
                        int dec_factor, int *num_colors, double *weightsOut) {
  if (dec_factor <= 0) {
    fprintf(stderr, "Decimation factor ( %d ) should be positive !\n", dec_factor);
    return -1;
  }
  dq_context *ctx = dq_default_context();
  DefaultLock lock;
  require_device(ctx);
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  const uint32_t dec = (uint32_t)dec_factor;
  const uint32_t samples = ((numRows + dec - 1) / dec) * ((numCols + dec - 1) / dec);
  *num_colors = 0;
  if (samples == 0) return 0;
  ctx->d_in.ensure(numPixels);
  ctx->d_pts0.ensure(samples);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, inPixels, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  reset_control(ctx);
  check_sampling(numPixels, numRows, numCols, dec);
  ctx->d_uniq.ensure(samples);
  hist_insert(ctx->d_in.ptr, numPixels, numRows, numCols, dec, 8, ctx->d_table, ctx->d_uniq.ptr, &ctx->d_cb->ucount,
              ctx->sm_count, ctx->stream);
  hist_collect(ctx->d_uniq.ptr, &ctx->d_cb->ucount, samples, ctx->d_table, ctx->d_pts0.ptr, true, ctx->sm_count, ctx->stream);
  DQ_CUDA_CHECK(cudaMemcpyAsync(&ctx->h_cb->ucount, &ctx->d_cb->ucount, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  const uint32_t U = ctx->h_cb->ucount;
  // emission order of the reference: (bucket asc, first-seen desc) keys, sorted, and the colours / weights written out in
  // that order -- all on the device; the host only copies the two result arrays back
  uint32_t n_pow2 = 2;
  while (n_pow2 < U) n_pow2 <<= 1;
  ctx->d_keys.ensure(n_pow2);
  ctx->d_out.ensure(std::max<size_t>(n_pow2, numPixels));                     // payload of the sort
  ctx->d_exact.ensure((size_t)U + 2);                                         // U doubles: the weights
  order_keys(ctx->d_in.ptr, numRows, numCols, dec, 8, ctx->d_uniq.ptr, ctx->d_pts0.ptr, U, ctx->d_table, ctx->d_keys.ptr,
             ctx->sm_count, ctx->stream);
  const double norm = sample_norm(numRows, numCols, dec_factor);
  uint32_t *d_colours = ctx->d_uniq.ptr;  // (the arrival-order list is not needed any more)
  double *d_weights = reinterpret_cast<double *>(ctx->d_exact.ptr);
  order_sort_emit(ctx->d_pts0.ptr, U, ctx->d_keys.ptr, ctx->d_out.ptr, norm, d_colours, d_weights, ctx->sm_count, ctx->stream);
  DQ_CUDA_CHECK(cudaMemcpyAsync(outPixels, d_colours, (size_t)U * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (weightsOut)
    DQ_CUDA_CHECK(cudaMemcpyAsync(weightsOut, d_weights, (size_t)U * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  *num_colors = (int)U;
  ctx->stats.num_points = U;
  return 0;
}

// ---- block majority vote ----

void dq_block_vote_device(dq_context *ctx, const uint32_t *d_quantPixels, uint32_t width, uint32_t height, uint32_t superpixelDim,
                          uint32_t *d_blocksOut) {
  require_device(ctx);
  if (superpixelDim < 1 || superpixelDim > 8 || width == 0 || height == 0) {
    fprintf(stderr, "divquant_b200: block vote needs a non-empty image and superpixelDim in 1..8\n");
    abort();
  }
  block_vote(d_quantPixels, width, height, superpixelDim, d_blocksOut, ctx->sm_count, ctx->stream);
  ctx->stats.kernel_launches++;
}

void dq_block_vote(const uint32_t *quantPixels, uint32_t width, uint32_t height, uint32_t superpixelDim, uint32_t *blocksOut) {
  if (superpixelDim < 1 || superpixelDim > 8 || width == 0 || height == 0) {
    fprintf(stderr, "divquant_b200: block vote needs a non-empty image and superpixelDim in 1..8\n");
    abort();
  }
  dq_context *ctx = dq_default_context();
  DefaultLock lock;
  require_device(ctx);
  const uint32_t n = width * height;
  const uint32_t nb = ((width + superpixelDim - 1) / superpixelDim) * ((height + superpixelDim - 1) / superpixelDim);
  ctx->d_in.ensure(n);
  ctx->d_out.ensure(n);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, quantPixels, (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  dq_block_vote_device(ctx, ctx->d_in.ptr, width, height, superpixelDim, ctx->d_out.ptr);
  DQ_CUDA_CHECK(cudaMemcpyAsync(blocksOut, ctx->d_out.ptr, (size_t)nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}

void dq_quant_blocks(const uint32_t *inPixels, uint32_t width, uint32_t height, uint32_t superpixelDim, const uint32_t *colortable,
                     int colormapSize, uint32_t *quantOut, uint32_t *blocksOut) {
  if (superpixelDim < 1 || superpixelDim > 8 || width == 0 || height == 0) {
    fprintf(stderr, "divquant_b200: block vote needs a non-empty image and superpixelDim in 1..8\n");
    abort();
  }
  dq_context *ctx = dq_default_context();
  DefaultLock lock;
  require_device(ctx);
  const uint32_t n = width * height;
  const uint32_t nb = ((width + superpixelDim - 1) / superpixelDim) * ((height + superpixelDim - 1) / superpixelDim);
  ctx->d_in.ensure(n);
  ctx->d_out.ensure(n);
  ctx->d_keys.ensure(nb / 2 + 2);  // 8-byte scratch reused for the nb block words
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, inPixels, (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  dq_map_colors_device(ctx, ctx->d_in.ptr, n, ctx->d_out.ptr, colortable, colormapSize, 1);
  uint32_t *d_blocks = reinterpret_cast<uint32_t *>(ctx->d_keys.ptr);
  dq_block_vote_device(ctx, ctx->d_out.ptr, width, height, superpixelDim, d_blocks);
  if (quantOut) DQ_CUDA_CHECK(cudaMemcpyAsync(quantOut, ctx->d_out.ptr, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaMemcpyAsync(blocksOut, d_blocks, (size_t)nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}

// ---- SRM front half ----

uint32_t dq_srm_num_pairs(uint32_t width, uint32_t height) { return srm_num_pairs(width, height); }

void dq_srm_sorted_edges_device(dq_context *ctx, const uint8_t *d_in, uint32_t width, uint32_t height, uint32_t channels,
                                uint32_t widthStep, dq_srm_pair *d_orderedPairs) {
  require_device(ctx);
  if (width == 0 || height == 0 || channels < 3 || widthStep < width * channels) {
    fprintf(stderr, "divquant_b200: SRM edges need a non-empty image with >= 3 interleaved channels and widthStep >= width*channels\n");
    abort();
  }
  ctx->d_keys.ensure(srm_scratch_words(width, height) / 2 + 2);
  ctx->stats.kernel_launches += srm_sorted_edges(d_in, width, height, channels, widthStep, reinterpret_cast<uint32_t *>(d_orderedPairs),
                                                 reinterpret_cast<uint32_t *>(ctx->d_keys.ptr), ctx->stream);
}

void dq_srm_sorted_edges(const uint8_t *in, uint32_t width, uint32_t height, uint32_t channels, uint32_t widthStep,
                         dq_srm_pair *orderedPairs) {
  dq_context *ctx = dq_default_context();
  DefaultLock lock;
  require_device(ctx);
  const size_t bytes = (size_t)height * widthStep;
  const uint32_t n = srm_num_pairs(width, height);
  ctx->d_in.ensure(bytes / 4 + 1);
  ctx->d_pts0.ensure(((size_t)n * 3 + 1) / 2 + 1);  // 8-byte elements holding the 12-byte pairs
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, in, bytes, cudaMemcpyHostToDevice, ctx->stream));
  dq_srm_pair *d_pairs = reinterpret_cast<dq_srm_pair *>(ctx->d_pts0.ptr);
  dq_srm_sorted_edges_device(ctx, reinterpret_cast<const uint8_t *>(ctx->d_in.ptr), width, height, channels, widthStep, d_pairs);
  DQ_CUDA_CHECK(cudaMemcpyAsync(orderedPairs, d_pairs, (size_t)n * sizeof(dq_srm_pair), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
}

// ---- label image ----

void dq_colortable_indexes_device(dq_context *ctx, const uint32_t *d_quantPixels, uint32_t numPixels, const uint32_t *colortable,
                                  int colormapSize, uint32_t *d_labelsOut, int asGreyscale) {
  require_device(ctx);
  if (colormapSize <= 0 || colormapSize > 24000) {
    fprintf(stderr, "divquant_b200: colortable of %d entries is not supported for label images (1..24000)\n", colormapSize);
    abort();
  }
  // colour -> last index holding it (the reference fills an unordered_map in palette order, :795-799)
  std::vector<std::pair<uint32_t, uint32_t>> pairs;
  pairs.reserve(colormapSize);
  for (int i = 0; i < colormapSize; ++i) pairs.emplace_back(colortable[i] & 0x00FFFFFFu, (uint32_t)i);
  std::stable_sort(pairs.begin(), pairs.end(), [](const std::pair<uint32_t, uint32_t> &a, const std::pair<uint32_t, uint32_t> &b) { return a.first < b.first; });
  std::vector<uint2> uniq;
  for (size_t i = 0; i < pairs.size(); ++i) {
    if (!uniq.empty() && uniq.back().x == pairs[i].first) uniq.back().y = pairs[i].second;  // later duplicate wins
    else uniq.push_back(make_uint2(pairs[i].first, pairs[i].second));
    if (asGreyscale && pairs[i].second > 255u) {
      fprintf(stderr, "divquant_b200: greyscale label images need indexes below 256\n");
      abort();  // assert(offset < 256) (:836)
    }
  }
  ctx->d_keys.ensure(uniq.size() + 1);  // reuse the 8-byte scratch buffer for the pairs
  reset_control(ctx);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_keys.ptr, uniq.data(), uniq.size() * sizeof(uint2), cudaMemcpyHostToDevice, ctx->stream));
  map_labels(d_quantPixels, numPixels, d_labelsOut, reinterpret_cast<const uint2 *>(ctx->d_keys.ptr), (int)uniq.size(), asGreyscale,
             &ctx->d_cb->ucount, ctx->sm_count, ctx->stream);
  DQ_CUDA_CHECK(cudaMemcpyAsync(&ctx->h_cb->ucount, &ctx->d_cb->ucount, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  if (ctx->h_cb->ucount != 0) {
    fprintf(stderr, "divquant_b200: pixel %u has no matching colortable entry\n", ctx->h_cb->ucount - 1);
    abort();  // assert(0) (:823)
  }
}

void dq_colortable_indexes(const uint32_t *quantPixels, uint32_t numPixels, const uint32_t *colortable, int colormapSize,
                           uint32_t *labelsOut, int asGreyscale) {
  if (numPixels == 0) return;
  dq_context *ctx = dq_default_context();
  DefaultLock lock;
  require_device(ctx);
  ctx->d_in.ensure(numPixels);
  ctx->d_out.ensure(numPixels);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, quantPixels, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  dq_colortable_indexes_device(ctx, ctx->d_in.ptr, numPixels, colortable, colormapSize, ctx->d_out.ptr, asGreyscale);
  DQ_CUDA_CHECK(cudaMemcpy(labelsOut, ctx->d_out.ptr, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyDeviceToHost));
}

// ---- frame pipeline ----

}  // extern "C"

// ---- frame pipeline: lanes ------------------------------------------------------------------------------------
// One frame's critical path is a chain of ~100 dependent passes inside the persistent split kernel, which keeps
// most of the GPU idle.  Frames are independent, so the pipeline runs `lanes` of them side by side: every lane
// owns a context (stream, tables, scratch) and a pair of frame buffers, and one host thread (pipeline_dispatcher)
// walks each lane's frames, one at a time, through H2D -> kernels -> D2H.  Split kernels of different lanes occupy
// disjoint groups of SMs (dq_context_set_split_ctas); histogram / remap kernels and the copy engines fill in around them.
struct dq_pipeline {
  struct Job {
    uint64_t ticket = 0;
    uint32_t n = 0;
    const uint32_t *in = nullptr;
    uint32_t *out = nullptr, *k_ptr = nullptr, *colortable = nullptr;
    int all_unique = 0;
    bool device_ptrs = false;
  };
  struct Lane {
    dq_context *ctx = nullptr;
    uint32_t *d_in = nullptr, *d_out = nullptr;
    cudaEvent_t begin = nullptr, end = nullptr;
    bool have_begin = false;
    cudaEvent_t done = nullptr;
    // dispatcher state
    int state = 0;
    Job job;
  };
  int device = 0;
  uint32_t max_pixels = 0;
  std::vector<Lane> lanes;
  std::mutex mu;
  std::condition_variable cv_work, cv_done;
  std::deque<Job> queue;
  std::set<uint64_t> done_above;  // completed tickets >= low_water
  uint64_t submitted = 0, low_water = 0;  // every ticket < low_water has completed
  bool stop = false;
  std::atomic<uint64_t> launches{0};
  std::atomic<uint64_t> flagged_frames{0};  // frames whose tie audit raised a flag
  std::atomic<uint64_t> resolved_frames{0};  // ... settled by the resolver / forced cuts (dq_call_stats::tie_resolved, cut_overrides)
  std::atomic<uint64_t> rerun_frames{0};     // ... computed again on the ordered path (dq_call_stats::ordered_rerun)
  int poll_sleep = 0;    // the dispatcher sleeps 20 us between polling rounds instead of spinning (dq_pipeline_set_blocking_wait)
  std::thread dispatcher;
  float last_ms = 0.f;
};

namespace {

// How the tie audit's recovery steps settled the frame the lane's context just finished (before pipeline_complete).
void pipeline_count_ties(dq_pipeline *p, const dq_context *ctx) {
  if (ctx->stats.tie_resolved || ctx->stats.cut_overrides) p->resolved_frames++;
  if (ctx->stats.ordered_rerun) p->rerun_frames++;
}

void pipeline_complete(dq_pipeline *p, uint64_t ticket, uint64_t launches) {
  p->launches += launches;
  {
    std::lock_guard<std::mutex> lock(p->mu);
    p->done_above.insert(ticket);
    while (!p->done_above.empty() && *p->done_above.begin() == p->low_water) {
      p->done_above.erase(p->done_above.begin());
      p->low_water++;
    }
  }
  p->cv_done.notify_all();
}

// The dispatcher: ONE host thread walks the frames of all lanes through the GPU.  A lane is a small state machine
//   idle -> [H2D] histogram + split queued -> (palette arrives in the lane's mailbox) host palette handling, remap [+ D2H]
//        queued -> (the lane's event fires) frame complete -> idle
// and the thread only ever polls: mailboxes are host memory, events are cudaEventQuery.  Nothing sleeps on the GPU and
// nothing spins per lane, so the pipeline needs one busy host core however many lanes it feeds (round 1
// had a spinning thread per lane, and lost a quarter of its throughput where ranks had fewer cores than lanes).
void pipeline_dispatcher(dq_pipeline *p) {
  require_device(p->lanes[0].ctx);
  enum { kIdle = 0, kWaitSplit = 1, kWaitDone = 2 };
  for (;;) {
    bool progress = false;
    int busy = 0;
    for (dq_pipeline::Lane &lane : p->lanes) {
      dq_context *ctx = lane.ctx;
      if (lane.state == kWaitDone) {
        if (cudaEventQuery(lane.done) == cudaErrorNotReady) {
          ++busy;
          continue;
        }
        progress = true;
        lane.state = kIdle;
        if (ctx->stats.tie_flags) p->flagged_frames++;
        pipeline_count_ties(p, ctx);
        pipeline_complete(p, lane.job.ticket, ctx->stats.kernel_launches);
      } else if (lane.state == kWaitSplit) {
        ++busy;
        if (!quantize_pending_ready(ctx)) continue;
        progress = true;
        const dq_pipeline::Job &job = lane.job;
        // (a frame the tie audit flagged comes back here once or twice more: resolver verdict, ordered re-run)
        if (quantize_step(ctx, job.k_ptr, job.colortable) != kQuantDone) continue;
        const uint32_t *d_in = job.device_ptrs ? job.in : lane.d_in;
        uint32_t *d_out = job.device_ptrs ? job.out : lane.d_out;
        recurse_remap_tail(ctx, job.n, d_in, d_out, job.k_ptr, job.colortable);
        if (!job.device_ptrs)
          DQ_CUDA_CHECK(cudaMemcpyAsync(job.out, lane.d_out, (size_t)job.n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        DQ_CUDA_CHECK(cudaEventRecord(lane.done, ctx->stream));
        DQ_CUDA_CHECK(cudaEventRecord(lane.end, ctx->stream));
        lane.state = kWaitDone;
      }
    }
    // new frames for the idle lanes
    for (dq_pipeline::Lane &lane : p->lanes) {
      if (lane.state != kIdle) continue;
      {
        std::lock_guard<std::mutex> lock(p->mu);
        if (p->queue.empty()) break;
        lane.job = p->queue.front();
        p->queue.pop_front();
      }
      progress = true;
      ++busy;
      dq_context *ctx = lane.ctx;
      const dq_pipeline::Job &job = lane.job;
      if (!lane.have_begin) {
        DQ_CUDA_CHECK(cudaEventRecord(lane.begin, ctx->stream));
        lane.have_begin = true;
      }
      const uint32_t *d_in = job.device_ptrs ? job.in : lane.d_in;
      if (!job.device_ptrs)
        DQ_CUDA_CHECK(cudaMemcpyAsync(lane.d_in, job.in, (size_t)job.n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
      memset(&ctx->stats, 0, sizeof(ctx->stats));
      ctx->stats.num_pixels = job.n;
      recurse_begin(ctx, job.n, d_in, *job.k_ptr, job.all_unique);
      lane.state = kWaitSplit;
    }
    if (progress) continue;
    if (busy == 0) {
      std::unique_lock<std::mutex> lock(p->mu);
      p->cv_work.wait(lock, [&] { return p->stop || !p->queue.empty(); });
      if (p->queue.empty()) return;  // stop requested and nothing left
    } else if (p->poll_sleep) {
      std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
  }
}

uint64_t pipeline_enqueue(dq_pipeline *p, uint32_t n, const uint32_t *in, uint32_t *out, uint32_t *k_ptr, uint32_t *colortable,
                          int all_unique, bool device_ptrs) {
  if (!device_ptrs && n > p->max_pixels) {
    fprintf(stderr, "divquant_b200: frame of %u pixels exceeds the pipeline's max_pixels (%u)\n", n, p->max_pixels);
    abort();
  }
  check_quant_args(n, *k_ptr, 8);
  dq_pipeline::Job job;
  job.n = n;
  job.in = in;
  job.out = out;
  job.k_ptr = k_ptr;
  job.colortable = colortable;
  job.all_unique = all_unique;
  job.device_ptrs = device_ptrs;
  {
    std::lock_guard<std::mutex> lock(p->mu);
    job.ticket = p->submitted++;
    p->queue.push_back(job);
  }
  p->cv_work.notify_one();
  return job.ticket;
}

}  // namespace

extern "C" {

dq_pipeline *dq_pipeline_create_lanes(int device, uint32_t max_pixels, int lanes, int split_ctas) {
  if (lanes < 1) lanes = 1;
  if (lanes > 16) lanes = 16;
  dq_pipeline *p = new dq_pipeline();
  p->max_pixels = max_pixels;
  p->lanes.resize(lanes);
  for (auto &lane : p->lanes) {
    lane.ctx = dq_context_create(device);
    p->device = lane.ctx->device;
    // Default SM partition: the split kernels of all lanes together hold 3/4 of the SMs; the rest stays free for the
    // histogram / remap kernels, which cannot share an SM with a split CTA (it owns the register file).  Measured at
    // 4K, 12 lanes, with the chunked histogram (tools/lanes_check.py, B200): 8 CTAs each 0.158 ms/frame, 9: 0.153,
    // 10: 0.154, 11: 0.156; 1080p K = 64: 8: 0.100, 9: 0.095, 10: 0.094, 11: 0.093.  Before the chunked histogram the
    // best was 8 CTAs (11/16): more split SMs left it too few free SMs to keep enough L2 atomics in flight.  With the
    // wide-job points kept in shared memory (B200, 1000 W; 4K, 960 frames, two runs): 12 lanes x 8 CTAs 0.129 ms/frame,
    // x 9: 0.128-0.129, x 10: 0.135-0.136; 16 x 6: 0.122-0.123, 16 x 7: 0.129.  The shorter split did not move the best
    // partition.
    if (split_ctas <= 0) split_ctas = std::max(split2_max_ctas(lane.ctx->sm_count, 256) * 3 / 4 / lanes, lanes > 1 ? 4 : 1);
    if (lanes == 1) split_ctas = 0;  // a single lane is a single call: all SMs
    dq_context_set_split_ctas(lane.ctx, split_ctas);
    if (max_pixels) {
      DQ_CUDA_CHECK(cudaMalloc(&lane.d_in, (size_t)max_pixels * sizeof(uint32_t)));
      DQ_CUDA_CHECK(cudaMalloc(&lane.d_out, (size_t)max_pixels * sizeof(uint32_t)));
    }
    DQ_CUDA_CHECK(cudaEventCreate(&lane.begin));
    DQ_CUDA_CHECK(cudaEventCreate(&lane.end));
    DQ_CUDA_CHECK(cudaEventCreateWithFlags(&lane.done, cudaEventBlockingSync | cudaEventDisableTiming));
  }
  p->dispatcher = std::thread(pipeline_dispatcher, p);
  return p;
}

void dq_pipeline_set_blocking_wait(dq_pipeline *p, int enabled) {
  dq_pipeline_flush(p);
  p->poll_sleep = enabled ? 1 : 0;
}

dq_pipeline *dq_pipeline_create(int device, uint32_t max_pixels, int depth) {
  if (depth < 2) depth = 2;
  if (depth > 8) depth = 8;
  return dq_pipeline_create_lanes(device, max_pixels, depth, 0);
}

void dq_pipeline_destroy(dq_pipeline *p) {
  if (!p) return;
  dq_pipeline_flush(p);
  {
    std::lock_guard<std::mutex> lock(p->mu);
    p->stop = true;
  }
  p->cv_work.notify_all();
  p->dispatcher.join();
  for (auto &lane : p->lanes) {
    require_device(lane.ctx);
    cudaFree(lane.d_in);
    cudaFree(lane.d_out);
    cudaEventDestroy(lane.begin);
    cudaEventDestroy(lane.end);
    cudaEventDestroy(lane.done);
    dq_context_destroy(lane.ctx);
  }
  delete p;
}

uint64_t dq_pipeline_submit(dq_pipeline *p, uint32_t numPixels, const uint32_t *inPixelsPtr, uint32_t *outPixelsPtr,
                            uint32_t *numClustersPtr, uint32_t *outColortablePtr, int allPixelsUnique) {
  return pipeline_enqueue(p, numPixels, inPixelsPtr, outPixelsPtr, numClustersPtr, outColortablePtr, allPixelsUnique, false);
}

uint64_t dq_pipeline_submit_device(dq_pipeline *p, uint32_t numPixels, const uint32_t *d_in, uint32_t *d_out,
                                   uint32_t *numClustersPtr, uint32_t *outColortablePtr, int allPixelsUnique) {
  return pipeline_enqueue(p, numPixels, d_in, d_out, numClustersPtr, outColortablePtr, allPixelsUnique, true);
}

void dq_pipeline_wait(dq_pipeline *p, uint64_t ticket) {
  std::unique_lock<std::mutex> lock(p->mu);
  p->cv_done.wait(lock, [&] { return ticket < p->low_water || p->done_above.count(ticket) != 0; });
}

void dq_pipeline_flush(dq_pipeline *p) {
  {
    std::unique_lock<std::mutex> lock(p->mu);
    p->cv_done.wait(lock, [&] { return p->low_water == p->submitted; });
  }
  // device time from the first lane that started to the last that finished (workers are idle now)
  require_device(p->lanes[0].ctx);
  float span = 0.f;
  bool any = false;
  for (auto &a : p->lanes) {
    if (!a.have_begin) continue;
    for (auto &b : p->lanes) {
      if (!b.have_begin) continue;
      float ms = 0.f;
      DQ_CUDA_CHECK(cudaEventElapsedTime(&ms, a.begin, b.end));
      span = std::max(span, ms);
      any = true;
    }
  }
  if (any) p->last_ms = span;
  for (auto &lane : p->lanes) lane.have_begin = false;
}

float dq_pipeline_last_elapsed_ms(const dq_pipeline *p) { return p->last_ms; }
dq_context *dq_pipeline_context(dq_pipeline *p) { return p->lanes[0].ctx; }
uint64_t dq_pipeline_kernel_launches(const dq_pipeline *p) { return p->launches.load(); }
uint64_t dq_pipeline_flagged_frames(const dq_pipeline *p) { return p->flagged_frames.load(); }
uint64_t dq_pipeline_resolved_frames(const dq_pipeline *p) { return p->resolved_frames.load(); }
uint64_t dq_pipeline_rerun_frames(const dq_pipeline *p) { return p->rerun_frames.load(); }
int dq_pipeline_lanes(const dq_pipeline *p) { return (int)p->lanes.size(); }

// ---- test hooks ----

uint32_t dq_debug_split_timeline(dq_context *ctx, int enable, uint64_t *pairs_out, uint32_t capacity_pairs) {
  require_device(ctx);
  ctx->trace_split = enable ? 1 : 0;
  if (!pairs_out || !ctx->d_timeline.ptr) return 0;
  unsigned long long n = 0;
  DQ_CUDA_CHECK(cudaMemcpy(&n, ctx->d_timeline.ptr, sizeof(n), cudaMemcpyDeviceToHost));
  if (n > capacity_pairs) n = capacity_pairs;
  DQ_CUDA_CHECK(cudaMemcpy(pairs_out, ctx->d_timeline.ptr + 1, (size_t)n * 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return (uint32_t)n;
}

uint32_t dq_debug_split_points(dq_context *ctx, const uint32_t *colours, const uint32_t *counts, uint32_t num_points,
                               double norm, uint32_t num_colors, int max_iters, int num_bits, uint32_t *colortable,
                               dq_split_record *records, double *cluster_mean, uint32_t *cluster_size) {
  require_device(ctx);
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  static_assert(sizeof(dq_split_record) == sizeof(SplitRecord), "record layouts must match");
  // host points, no histogram: unweighted (no tie audit), and with records requested no mailbox
  dq_context::QuantState &q = ctx->qs;
  q = dq_context::QuantState();
  q.n = num_points, q.K = num_colors, q.point_cap = num_points;
  q.num_bits = num_bits, q.max_iters = max_iters, q.norm = norm;
  q.records = records, q.mean_out = cluster_mean, q.size_out = cluster_size;
  std::vector<uint2> pts(num_points);
  for (uint32_t i = 0; i < num_points; ++i) pts[i] = make_uint2(colours[i] & 0x00FFFFFFu, counts ? counts[i] : 1u);
  ctx->d_pts0.ensure(num_points);
  reset_control(ctx);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_pts0.ptr, pts.data(), (size_t)num_points * sizeof(uint2), cudaMemcpyHostToDevice, ctx->stream));
  ctx->h_cb->ucount = num_points;
  DQ_CUDA_CHECK(cudaMemcpyAsync(&ctx->d_cb->ucount, &ctx->h_cb->ucount, sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  plan_paths(ctx);
  run_split(ctx, SplitRun::kFirst);
  return run_split_finish(ctx, colortable);
}

uint32_t dq_debug_histogram(dq_context *ctx, const uint32_t *inPixels, uint32_t numPixels, uint32_t *colours, uint32_t *counts) {
  require_device(ctx);
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  if (numPixels == 0) return 0;
  ctx->d_in.ensure(numPixels);
  ctx->d_pts0.ensure(numPixels);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, inPixels, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  reset_control(ctx);
  run_histogram(ctx, ctx->d_in.ptr, numPixels, 1, numPixels, 1, 8);
  hist_collect(ctx->d_uniq.ptr, &ctx->d_cb->ucount, numPixels, ctx->d_table, ctx->d_pts0.ptr, true, ctx->sm_count, ctx->stream);
  DQ_CUDA_CHECK(cudaMemcpyAsync(&ctx->h_cb->ucount, &ctx->d_cb->ucount, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  const uint32_t U = ctx->h_cb->ucount;
  std::vector<uint2> pts(U);
  DQ_CUDA_CHECK(cudaMemcpy(pts.data(), ctx->d_pts0.ptr, (size_t)U * sizeof(uint2), cudaMemcpyDeviceToHost));
  for (uint32_t i = 0; i < U; ++i) {
    colours[i] = pts[i].x;
    counts[i] = pts[i].y;
  }
  ctx->stats.num_points = U;
  return U;
}

uint32_t dq_pixel_histogram(const uint32_t *pixels, uint32_t numPixels, uint32_t *pixelsOut, uint32_t *countsOut, uint32_t capacity) {
  dq_context *ctx = dq_default_context();
  DefaultLock lock;
  require_device(ctx);
  if (numPixels == 0) return 0;
  ctx->d_in.ensure(numPixels);
  ctx->d_pts0.ensure(numPixels);
  DQ_CUDA_CHECK(cudaMemcpyAsync(ctx->d_in.ptr, pixels, (size_t)numPixels * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  reset_control(ctx);
  run_histogram(ctx, ctx->d_in.ptr, numPixels, 1, numPixels, 1, 8);
  hist_collect(ctx->d_uniq.ptr, &ctx->d_cb->ucount, numPixels, ctx->d_table, ctx->d_pts0.ptr, true, ctx->sm_count, ctx->stream);
  DQ_CUDA_CHECK(cudaMemcpyAsync(&ctx->h_cb->ucount, &ctx->d_cb->ucount, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  const uint32_t U = ctx->h_cb->ucount;
  std::vector<uint2> pts(U);
  DQ_CUDA_CHECK(cudaMemcpy(pts.data(), ctx->d_pts0.ptr, (size_t)U * sizeof(uint2), cudaMemcpyDeviceToHost));
  std::sort(pts.begin(), pts.end(), [](const uint2 &a, const uint2 &b) { return a.x < b.x; });
  for (uint32_t i = 0; i < U && i < capacity; ++i) {
    pixelsOut[i] = pts[i].x;
    countsOut[i] = pts[i].y;
  }
  return U;
}

}  // extern "C"

// ---- pixel-row sharding of one image, exchange inside the library (NCCL) ---------------------------------------------
// BASELINE config 3.  Every rank histograms its own rows; the per-shard (colour, count, first-seen index) lists are
// exchanged with ONE grouped ncclAllGather on the context's stream (fixed-capacity slices, unused entries carry count 0, so
// no sizes have to travel first and nothing waits on the host); every rank merges the lists into its direct table (and the
// whole image's first-seen indexes into d_map, for the tie resolver) and runs the split replicated -- exact integer sums:
// identical decisions from identical integers on every GPU, flagged frames through quantize_step -- and remaps its own rows.
// NCCL is looked up at run time (dlopen of libnccl.so.2: the copy the process already has, e.g. PyTorch's, or the
// system's), so the library itself has no link-time dependency on it.
#include <dlfcn.h>
#include <nccl.h>

namespace {

struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
};

NcclApi *nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
      fprintf(stderr, "divquant_b200: the row-sharded path needs NCCL (libnccl.so.2 not found: %s)\n", dlerror());
      abort();
    }
    auto sym = [&](const char *name) {
      void *p = dlsym(h, name);
      if (!p) {
        fprintf(stderr, "divquant_b200: %s missing from libnccl\n", name);
        abort();
      }
      return p;
    };
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
    api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
    api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
    api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
  });
  return &api;
}

void nccl_check(ncclResult_t r, const char *what) {
  if (r != ncclSuccess) {
    fprintf(stderr, "divquant_b200: NCCL error in %s: %s\n", what, nccl_api()->GetErrorString(r));
    abort();
  }
}

}  // namespace

struct dq_rows {
  dq_context *ctx = nullptr;
  ncclComm_t comm = nullptr;
  int world = 1, rank = 0;
  uint32_t cap = 0;              // list entries per rank
  uint32_t *d_colours = nullptr;  // [world][cap]
  uint32_t *d_counts = nullptr;   // [world][cap]
  uint32_t *d_first = nullptr;    // [world][cap + 1]: shard-local first-seen index of every listed colour, then the shard's pixels
  uint32_t *d_overflow = nullptr;
};

extern "C" {

void dq_rows_unique_id(void *out128) {
  ncclUniqueId id;
  nccl_check(nccl_api()->GetUniqueId(&id), "ncclGetUniqueId");
  memcpy(out128, &id, sizeof(id));
}

dq_rows *dq_rows_create(dq_context *ctx, int world, int rank, const void *unique_id128, uint32_t list_capacity) {
  require_device(ctx);
  if (world < 1 || rank < 0 || rank >= world || list_capacity == 0) {
    fprintf(stderr, "divquant_b200: dq_rows_create needs 0 <= rank < world and a positive list capacity\n");
    abort();
  }
  if ((uint64_t)world * ((uint64_t)list_capacity + 1) > 0xFFFFFFFFull) {  // (list offsets and entry counts are 32-bit)
    fprintf(stderr, "divquant_b200: dq_rows_create: world x (list_capacity + 1) must stay below 2^32\n");
    abort();
  }
  dq_rows *r = new dq_rows();
  r->ctx = ctx;
  r->world = world;
  r->rank = rank;
  r->cap = list_capacity;
  if (world > 1) {
    ncclUniqueId id;
    memcpy(&id, unique_id128, sizeof(id));
    nccl_check(nccl_api()->CommInitRank(&r->comm, world, id, rank), "ncclCommInitRank");
  }
  DQ_CUDA_CHECK(cudaMalloc(&r->d_colours, (size_t)world * list_capacity * sizeof(uint32_t)));
  DQ_CUDA_CHECK(cudaMalloc(&r->d_counts, (size_t)world * list_capacity * sizeof(uint32_t)));
  DQ_CUDA_CHECK(cudaMalloc(&r->d_first, (size_t)world * (list_capacity + 1) * sizeof(uint32_t)));
  DQ_CUDA_CHECK(cudaMalloc(&r->d_overflow, sizeof(uint32_t)));
  DQ_CUDA_CHECK(cudaMemset(r->d_overflow, 0, sizeof(uint32_t)));
  return r;
}

void dq_rows_destroy(dq_rows *r) {
  if (!r) return;
  require_device(r->ctx);
  cudaStreamSynchronize(r->ctx->stream);
  if (r->comm) nccl_api()->CommDestroy(r->comm);
  cudaFree(r->d_colours);
  cudaFree(r->d_counts);
  cudaFree(r->d_first);
  cudaFree(r->d_overflow);
  delete r;
}

void dq_rows_quant_recurse(dq_rows *r, const uint32_t *d_shard, uint32_t n_shard, uint64_t total_pixels, uint32_t *d_out_shard,
                           uint32_t *numClustersPtr, uint32_t *outColortablePtr) {
  dq_context *ctx = r->ctx;
  require_device(ctx);
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  ctx->stats.num_pixels = n_shard;
  const uint32_t K = *numClustersPtr;
  if (total_pixels == 0 || total_pixels > 0x7fffffffull || K == 0) {
    fprintf(stderr, "divquant_b200: row-sharded call needs 0 < total_pixels < 2^31 and K > 0\n");
    abort();
  }
  const uint32_t cap = r->cap;
  const size_t entries = (size_t)r->world * cap;
  uint32_t *my_colours = r->d_colours + (size_t)r->rank * cap, *my_counts = r->d_counts + (size_t)r->rank * cap;
  uint32_t *my_first = r->d_first + (size_t)r->rank * (cap + 1);
  // 1. this rank's rows -> (colour, count, first-seen index) list in its slice (an empty shard is a list of zero counts)
  reset_control(ctx);
  ctx->d_pts0.ensure(std::max<size_t>(n_shard, entries));
  ctx->d_uniq.ensure(std::max<size_t>(n_shard, entries));
  if (n_shard) {
    hist_insert(d_shard, n_shard, 1, n_shard, 1, 8, ctx->d_table, ctx->d_uniq.ptr, &ctx->d_cb->ucount, ctx->sm_count, ctx->stream,
                ctx->d_map);
    first_seen_launch(exact_sampling(d_shard, 1, n_shard, 1, 8), ctx->d_map, ctx->stream);
    hist_collect(ctx->d_uniq.ptr, &ctx->d_cb->ucount, n_shard, ctx->d_table, ctx->d_pts0.ptr, true, ctx->sm_count, ctx->stream);
    ctx->stats.kernel_launches += 3;
  }
  hist_export_padded(ctx->d_pts0.ptr, &ctx->d_cb->ucount, cap, my_colours, my_counts, r->d_overflow, ctx->sm_count, ctx->stream,
                     ctx->d_map, my_first, n_shard);
  ctx->stats.kernel_launches++;
  // 2. the one exchange of the data path
  if (r->world > 1) {
    NcclApi *nc = nccl_api();
    nccl_check(nc->GroupStart(), "ncclGroupStart");
    nccl_check(nc->AllGather(my_colours, r->d_colours, cap, ncclUint32, r->comm, ctx->stream), "ncclAllGather(colours)");
    nccl_check(nc->AllGather(my_counts, r->d_counts, cap, ncclUint32, r->comm, ctx->stream), "ncclAllGather(counts)");
    nccl_check(nc->AllGather(my_first, r->d_first, cap + 1, ncclUint32, r->comm, ctx->stream), "ncclAllGather(first-seen)");
    nccl_check(nc->GroupEnd(), "ncclGroupEnd");
  }
  // 3. merged histogram (and first-seen indexes) of the whole image in this rank's direct table, split replicated with the
  //    tie audit's resolver and forced cuts (quantize_step), own rows remapped
  dq_context::QuantState &q = ctx->qs;
  q = dq_context::QuantState();
  q.merged.colours = r->d_colours, q.merged.counts = r->d_counts, q.merged.first = r->d_first;
  q.merged.cap = cap, q.merged.world = (uint32_t)r->world;
  q.n = (uint32_t)total_pixels, q.rows = 1, q.cols = (uint32_t)total_pixels, q.K = K, q.point_cap = (uint32_t)entries;
  q.norm = sample_norm(1, (uint32_t)total_pixels, 1);  // 1 / N of the WHOLE image (:172)
  q.table_dirty = true;
  quantize_launch(ctx);
  uint32_t k = K;
  quantize_finish(ctx, &k, outColortablePtr);
  // every colour of this rank's rows is in the merged list, so the table path serves the shard
  remap_quantized(ctx, n_shard, d_shard, d_out_shard, &k, outColortablePtr, true);
  *numClustersPtr = k;
  uint32_t overflow = 0;
  DQ_CUDA_CHECK(cudaMemcpyAsync(&overflow, r->d_overflow, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  DQ_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
  if (overflow) {
    fprintf(stderr, "divquant_b200: a shard has %u unique colours, more than the %u entries per rank the row exchange was created with\n",
            overflow, cap);
    abort();
  }
}

}  // extern "C"

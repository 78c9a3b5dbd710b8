// dq_split.cuh -- data structures of the divisive (variance split + local 2-means) phase.
//
// Reference: DivQuantCluster<UW,MT,KM>, DivQuant/DivQuantCluster.cpp:133-1097.
//
// The reference performs K-1 data-dependent splits one after another.  What a split produces
// (the two child centres, weights, variances, TSEs and point sets) is a pure function of the
// split cluster's own points and of the (weight, mean, variance) it inherited when it was created;
// only WHICH clusters get split, and the index each child receives, depend on the global
// max-TSE priority (:876-887).  The device therefore keeps a binary tree of "nodes":
//   * every round splits a batch of leaves at once (one persistent kernel, grid barriers between
//     the 1 + max_iters dependent passes of a round);
//   * a scalar "controller" (CTA 0) replays the reference's sequential selection over the cached
//     split results, stalls when it needs a split that has not been computed yet, and requests the
//     stalled leaf plus the leaves whose TSE rank is within the remaining split budget.
// Sums over points are exact u64 integer sums of count*c (and count*c*c); the reference's scalar
// formulas are then evaluated in IEEE double without FMA contraction, in the reference's order.
#pragma once

#include "dq_common.cuh"

namespace dq {

constexpr int kSplitThreads = 1024;  // one CTA per SM
constexpr int kSplitTile = 1024;     // points per tile (unit of work distribution)
constexpr int kSplitMaxIters = 32;   // the reference ships max_iters = 10 (quant_util.cpp:31)
constexpr int kAccWords = 8;         // per (job, pass): cnt, sumR, sumG, sumB, npts, sumRR, sumGG, sumBB

enum AccSlot { kAccCnt = 0, kAccR = 1, kAccG = 2, kAccB = 3, kAccPts = 4, kAccRR = 5, kAccGG = 6, kAccBB = 7 };

// A cluster at some moment of the reference's sequence.
struct SplitNode {
  double tw;      // total weight            (weight[], :293)
  double tm[3];   // componentwise mean      (mean[],   :316)
  double tv[3];   // componentwise variance  (var[],    :322)
  double tse;     // total squared error     (tse[],    :310)
  double cut;     // cutting position chosen when this node was scheduled for a split
  uint32_t begin; // its points are pts[buf][begin .. begin+size)
  uint32_t size;  // number of unique-colour points
  int32_t buf;
  int32_t child;  // node id of the "old" child (the "new" child is child+1); -1 = not split yet
  int32_t axis;   // cutting axis chosen when scheduled
  int32_t parent; // node this one was split from (-1 for the root)
  // Tie audit of the exact-integer path (dq_tie.cuh): first-order bounds on |this kernel's value - the reference's value|
  // of the three sums behind the statistics (W, S = W*mean, Q = W*(var + mean^2)) and, derived from them, of tm[], tv[]
  // and tse; and the decisions of this node's own split that fell inside such a bound (TieBit mask).
  double eW, eS, eQ, eM, eV, eT;
  uint32_t tie;
  uint32_t pad;
};

// A split being computed in the current round.
struct SplitJob {
  double cut;
  double tw;
  double tm[3];
  int32_t node;
  int32_t axis;
  uint32_t begin;
  uint32_t size;
  int32_t buf;
  uint32_t tile0;    // first tile of this job in the round's tile numbering
  uint32_t cur_old;  // scatter cursors of the partition pass (relative to the child segment)
  uint32_t cur_new;
  int32_t child0;    // node id reserved for the "old" child (child0+1 = "new" child)
  int32_t pad;
};

// Mirrors oracle_split_record (oracle/divquant_oracle.h) so tests can compare field by field.
struct SplitRecord {
  int32_t new_index, old_index, cut_axis, num_points, new_size, is_last;
  double cut_pos;
  double total_weight, new_weight, old_weight;
  double new_mean[3], old_mean[3];
  double new_var[3], old_var[3];
  double new_tse, old_tse;
};

// timeline tags
enum TraceTag { kTraceRoundBegin = 1, kTracePhaseA = 2, kTracePhaseB = 3, kTracePhaseC = 4, kTraceCtlBarrier = 5, kTracePass = 6, kTracePartition = 7, kTraceRoot = 8, kTraceBegin = 9, kTraceCollected = 10, kTraceReduced = 11, kTraceRootBarrier = 12, kTraceNarrowJob = 13 };

enum CtlSlot {
  kCtlJobs = 0,    // jobs in the current round
  kCtlTiles = 1,   // tiles in the current round
  kCtlDone = 2,    // 1 when the controller has finished
  kCtlNodes = 3,   // nodes allocated so far
  kCtlRounds = 4,  // rounds executed (diagnostics)
  kCtlSplits = 5,  // splits computed, including speculative ones (diagnostics)
  kCtlError = 6,   // non-zero = internal inconsistency
  kCtlTie = 8,     // tie audit: TieBit mask of the decisions that sit inside the reference's rounding noise (dq_tie.cuh)
  kCtlTieCount = 9,  // tie audit: final clusters whose palette rounding is flagged (entries of SplitArgs::tie_list)
  kCtlCutCount = 10,  // tie audit: consumed splits whose cut is flagged (entries of the second list of tie_list)
  kCtlWords = 12   // [kCtlWords - 1] = detail of an expired wait
};

// Decisions of the divisive phase that the exact-integer sums may take differently from the reference's sequential
// double sums (DESIGN.md 5.2): bit d-1 = decision kind d was found inside the noise bound somewhere in the frame.
enum TieBit {
  kTieAxis = 1u,        // D1: two channel variances of a split cluster (:388-403)
  kTieCut = 2u,         // D2: cut_pos < proj_val (:473)
  kTieHyperplane = 4u,  // D3: lhs < rhs . x (:683)
  kTieTse = 8u,         // D4: arg-max of the TSEs (:876-887), incl. the DBL_MIN seed
  kTieRound = 16u,      // D5: (uint8)(mean + 0.5) (:1050-1052)
  kTieReplay = 32u,     // the sequential replay of the selection ran (degenerate TSE order): not audited, always flagged
  kTieUnaudited = 64u   // set by the host: exact-integer sums WITHOUT an audit (K > kSplit2MaxColors beyond the ordered path)
};

struct CutOverride {
  uint32_t begin, size;
  double mean_here, mean_ref;
};
constexpr uint32_t kCutOverrideCap = 16;

struct SplitArgs {
  uint2 *pts[2];        // (colour 0x00RRGGBB, count) double buffer, capacity U each
  uint32_t num_points;  // U (ignored when num_points_dev != nullptr)
  const uint32_t *num_points_dev;  // U produced on the device by the histogram
  uint32_t num_colors;  // requested K
  int32_t max_iters;    // >= 1
  int32_t shift;        // 8 - num_bits
  double norm;          // 1 / #sampled pixels  (data_weight / norm_factor)
  SplitNode *nodes;
  uint32_t node_cap;
  SplitJob *jobs;       // [2][K], double-buffered by round parity
  uint64_t *acc;        // [2][K][max_iters+1][kAccWords]
  uint64_t *root_acc;   // [kAccWords]
  uint32_t *ctl;        // [kCtlWords]
  unsigned int *barrier;
  // controller arrays in global memory, used when they do not fit in shared memory
  int32_t *g_cluster_node;  // [K]
  double *g_cluster_tse;    // [K]
  int32_t use_smem_ctl;
  // outputs
  uint32_t *palette;      // [K]   non-empty clusters in index order (:1030-1065)
  uint32_t *result;       // [0] = number of clusters emitted, [1] = number of empty clusters
  double *cluster_mean;   // [K][3]   (diagnostics / tests)
  uint32_t *cluster_size; // [K]
  SplitRecord *records;   // [K-1] or nullptr
  // optional trace: CTA 0 appends (tag, SM clock) pairs; [0] = number of pairs (tracing aid, see tools/)
  unsigned long long *timeline;
  uint32_t timeline_cap;
  // Optional host mailbox (mapped pinned memory): when the kernel has finished, CTA 0 stores
  //   [1] U  [2..5] result  [6..13] ctl  [16..16+K) palette, a system fence, then [0] = mailbox_seq,
  // so the host can poll for the palette instead of waiting for the stream and copying it (dq_split2.cu only).
  uint32_t *mailbox;
  uint32_t mailbox_seq;
  // inputs of at most this many points are handled by split_exact_kernel (dq_split_exact.cu): the split kernels
  // return at once for them.  0 = off.
  uint32_t exact_small_max;
  // 1 = weighted path on exact-integer sums: audit every decision against the reference's rounding noise (dq_tie.cuh)
  uint32_t tie_audit;
  // final clusters flagged kTieRound: {cluster index, node id, palette slot, 0} each, at most kTieListCap (dq_resolve.cu)
  uint32_t *tie_list;
  // SM cycles a wait on another CTA may last before it is declared stuck (0 = the built-in 0.2 s)
  long long spin_cycles;
  // Cuts taken from the resolver (dq_resolve.cu): a node whose range is [begin, begin + size) and whose own mean on the cut
  // axis is exactly `mean_here` is cut at `mean_ref`, the mean the reference holds for it, and its cut is not audited again.
  const CutOverride *cut_overrides;
  uint32_t num_cut_overrides;
};
constexpr uint32_t kTieListCap = 16;
// layout of the tie_list buffer (words): [0, 4 cap) rounding entries | [4 cap, 6 cap) resolver status, roundings then cuts |
// [6 cap, 6 cap + 4) a counter of the resolver | [kTieCutList, + cap) nodes whose cut is flagged
constexpr uint32_t kTieStatus = 4 * kTieListCap, kTieCounter = 6 * kTieListCap, kTieCutList = 6 * kTieListCap + 4;
// [kTieRefCut, + 6 cap) one CutOverride per cut entry, written by the resolver (8-byte aligned offset)
constexpr uint32_t kTieRefCut = kTieCutList + kTieListCap;
static_assert(kTieRefCut % 2 == 0 && sizeof(CutOverride) == 24, "records with doubles inside the tie_list buffer");
constexpr uint32_t kTieListWords = kTieRefCut + 6 * kTieListCap;


// Largest input (unique colours) that takes the sequential-order path of dq_split_exact.cu.
constexpr uint32_t kExactMaxPoints = 262144;       // compile-time ceiling; the run-time limit is SplitArgs::exact_small_max
// Its default.  Above it the exact-integer kernels run with the tie audit (dq_tie.cuh) and only flagged frames come back
// to the ordered path; 4096 is where the ordered path stops being the cheaper way to be right: up to there ties are the
// rule (tiny clusters) and the whole input sits in shared memory (~1 ms); at 40 000 colours it costs 20 ms against 0.35.
// (36 natural crops of 4 000..60 000 colours, tools/limit_check.py: limit 65536 3.3 ms per crop, 4096 1.3 ms, all
// bit-exact either way.)
constexpr uint32_t kExactDefaultPoints = 4096;
constexpr uint32_t kExactMaxColors = 4096;
// Small weighted inputs in the reference's own summation order (dq_split_exact.cuh).
// The sampled pixels behind the histogram: needed to put the unique colours into calc_color_table's emission order.
struct ExactSampling {
  const uint32_t *in;
  uint32_t samples_per_row, num_samples, num_rows, dec, word_mask, shift;
};
ExactSampling exact_sampling(const uint32_t *d_in, uint32_t num_rows, uint32_t num_cols, uint32_t dec, int bits);
// dq_resolve.cu: a final cluster's mean in the reference's own arithmetic (ordered sums along its chain of splits), for the
// clusters whose rounding the tie audit flagged (n_round entries) and the nodes whose cut it flagged (n_cut entries).
// d_status[i]: 1 = settled (palette[slot] rewritten / the cut separates the same points), 2 = not resolvable here,
// 3 = the reference cuts this node differently.
void tie_resolve_launch(const SplitNode *d_nodes, uint32_t num_nodes, uint2 *const *pts, const uint32_t *d_first_seen, double norm,
                        int shift, const uint32_t *d_list, uint32_t n_round, uint32_t n_cut, uint32_t *d_palette, uint32_t *d_status,
                        cudaStream_t st);
// The same for chains through nodes of any size (global sort of the points under the top nodes, one streaming pass).
// Scratch: d_keys / d_vals hold the power of two >= u entries, d_flat u points, d_counter one word.
void tie_resolve_big_launch(const SplitNode *d_nodes, uint32_t num_nodes, uint2 *const *pts, const uint32_t *d_first_seen, uint32_t u,
                            double norm, int shift, const uint32_t *d_list, uint32_t n_round, uint32_t n_cut, uint64_t *d_keys,
                            uint32_t *d_vals, uint2 *d_flat, uint32_t *d_counter, uint32_t *d_palette, uint32_t *d_status,
                            int sm_count, cudaStream_t st);
// first-seen pass alone (dq_split_exact.cu): smallest sample index of every colour into d_first_seen
void first_seen_launch(const ExactSampling &q, uint32_t *d_first_seen, cudaStream_t st);
size_t split_exact_smem_bytes();
size_t split_exact_scratch_bytes();  // global scratch for the point arrays of inputs above 4096 colours
// Stand-alone form (two launches that return at once for large inputs).  g_f64: 8*K doubles, g_i32: K ints of scratch.
void split_exact_launch(const SplitArgs &args, const ExactSampling &q, unsigned char *d_scratch, const uint32_t *d_uniq,
                        uint32_t *d_table, uint32_t *d_first_seen, double *g_f64, int32_t *g_i32, cudaStream_t st);

constexpr int kMailboxPalette = 32;                      // word offset of the palette inside the mailbox
constexpr int kMailboxWords = kMailboxPalette + 512;     // K <= kSplit2MaxColors

// Launch description computed on the host.
struct SplitLaunch {
  int grid;
  size_t smem_bytes;
};

// v1: generic kernel (any K; controller on CTA 0, one grid barrier per pass)
SplitLaunch split_plan(int sm_count, uint32_t num_colors);
void split_launch(const SplitArgs &args, const SplitLaunch &plan, cudaStream_t stream);
size_t split_acc_words(uint32_t num_colors, int max_iters);

// v2: latency-optimised kernel (K <= kSplit2MaxColors): replicated controller, CTA-local narrow jobs,
// tag-in-data exchange of partial sums for wide jobs.  See dq_split2.cu.
constexpr uint32_t kSplit2MaxColors = 512;
struct Split2Extra {
  unsigned long long *slots;  // [2][slot_cap][kAccWords] tagged words, zeroed by the kernel
  uint32_t slot_cap;
  uint32_t *cursors;          // (unused since the partition takes its destinations from the exchanged counts)
  uint32_t *progress;         // [grid] last stage each CTA reached (diagnostics of an expired wait)
  // when non-null the root pass also builds the points from the histogram (fused hist_collect):
  // pts[0][i] = (uniq[i], table[uniq[i]]) and the counter is zeroed
  const uint32_t *collect_uniq;
  uint32_t *collect_table;
  // when exact_fused != 0 (and SplitArgs::exact_small_max != 0) the kernel itself handles small inputs: every CTA
  // takes part in the first-seen pass, then CTA 0 runs split_exact_body on the histogram above
  uint32_t exact_fused;
  ExactSampling exact_src;
  uint32_t *exact_first_seen;
  unsigned char *exact_scratch;  // split_exact_scratch_bytes()
  double *exact_f64;   // 8*K doubles
  int32_t *exact_i32;  // K ints
  // points of a CTA's wide-job shares that the round's cut pass keeps in the dynamic shared memory behind the integer path's
  // arrays, so that its later passes and the partition do not read them from L2 again (set by split2_launch from the plan)
  uint32_t wide_cache_points;
};
size_t split2_slot_capacity(uint32_t point_capacity, uint32_t num_colors, int sm_count);
SplitLaunch split2_plan(int requested_ctas, int sm_count, uint32_t num_colors);
int split2_max_ctas(int sm_count, uint32_t num_colors);
void split2_launch(const SplitArgs &args, const Split2Extra &extra, const SplitLaunch &plan, cudaStream_t stream);

}  // namespace dq

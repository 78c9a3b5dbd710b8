// dq_split2.cu -- latency-optimised divisive phase (K <= kSplit2MaxColors), one persistent
// cooperative sm_100a kernel.
//
// Reference: DivQuantCluster, DivQuant/DivQuantCluster.cpp:133-1097 (same formulation as dq_split.cu:
// a tree of speculatively computed splits + an exact replay of the reference's max-TSE sequence).
// What is different from the generic kernel is how the dependency chain is kept short:
//
//  * Replicated controller.  Every CTA keeps the whole controller state (TSE, child, size, parent of
//    every node) in its own shared memory and takes the same decisions from the same data, so a round
//    needs ONE grid barrier and no broadcast.
//  * Threshold policy instead of a sequential replay per round.  The reference pops the max-TSE leaf
//    K-1 times; since a child's TSE is below its parent's, the popped set is the K-1 largest TSEs of
//    the tree.  A leaf is therefore worth splitting only while fewer than K-1 known nodes have a larger
//    TSE -- a fully parallel test.  The exact sequence (cluster numbering, DBL_MIN / stale-index quirks)
//    is reconstructed once at the end: in parallel when the TSE order is strict (verified), otherwise
//    by the reference's sequential scan, replicated in every CTA (which may request more splits).
//  * Narrow jobs (<= 4096 points) run entirely inside one CTA: points live in registers for all
//    1 + max_iters passes, reductions are warp shuffles + shared memory, no global traffic.
//  * Wide jobs span many CTAs.  Partial sums are exchanged through per-(job, CTA) slots of 8-byte
//    words that carry their own 16-bit pass tag next to the 48-bit value, so publishing is a plain
//    store and gathering is one polling L2 read: no atomics, no fences, no barrier per pass.  The round's wide
//    tiles are dealt to the CTAs in contiguous blocks, so a job spans as few CTAs as possible and the partition --
//    whose destinations come from the participants' counts in those slots, not from atomics -- keeps tile order.
//  * Inputs small enough for the reference's own summation order leave at the top of the kernel into
//    dq_split_exact.cuh / dq_split_ordered.cuh (same launch, no host decision).
#include <cfloat>
#include <map>
#include <mutex>

#include "dq_split_exact.cuh"
#include "dq_split_math.cuh"

namespace dq {
namespace {

constexpr int kWarps = 16;
constexpr int T = 32 * kWarps;  // 16 warps, up to 128 registers per thread: points stay in registers without spills
constexpr uint32_t kWideTile = 1024;  // points per wide tile
constexpr int kNarrowPPT = 8;         // points per thread of a narrow job (kept in registers for all passes)
constexpr uint32_t kNarrowMax = kNarrowPPT * T;
constexpr int kGroupWarps = 8;                 // warps of a narrow-job group
constexpr int kGroups = kWarps / kGroupWarps;  // narrow jobs a CTA runs side by side
constexpr int kGroupT = 32 * kGroupWarps;
constexpr uint32_t kGroupMax = kNarrowPPT * kGroupT;  // largest narrow job a group holds in registers
constexpr int kWideCache = 4;         // wide jobs whose constants a CTA keeps in shared memory
constexpr unsigned long long kValueMask = (1ull << 48) - 1ull;

struct JobConst {
  double tw, tm[3], cut;
  int32_t axis, buf;
  uint32_t begin, size;
};
// Tie audit: what the bounds of a job's passes need from its node (dq_tie.cuh).  Lives in shared memory only; warp 1 and
// thread 0 read it, nobody keeps it in registers.  eM < 0 = audit off.
struct JobAudit {
  double eW, eS, eM, m1;  // m1 = max |tm_c|
};
constexpr int kAudCache = 32;  // wide jobs of a CTA whose audit constants are kept (more than that: flagged wholesale)

// A narrow job in flight in a group of kGroupWarps warps: the fields of Shared2 that one narrow job uses, under the same names.
struct NarrowGroup {
  uint64_t red[kGroupWarps][kAccWords];
  uint64_t tot[kAccWords];
  PassParams pp;
  tie::PassExt ext;
  JobAudit aud;
  SplitNode cur;
  uint64_t prev_tot[4];
  int32_t converged;
  uint32_t near, job_tie, cur_old, cur_new;
  int32_t next;  // the group's next entry of mynarrow
};

struct Shared2 {
  uint64_t red[32][kAccWords];
  uint64_t tot[kAccWords];
  PassParams pp;
  SplitNode root;
  SplitNode cur;  // node being split by a narrow job / finalised by an owner
  JobConst wide[kWideCache];
  PassParams wide_pp[kWideCache];  // classification of the last pass, reused by the partition
  uint32_t part_new[kWarps], part_old[kWarps], base_new, base_old;  // partition of wide jobs: offsets without atomics
  uint32_t piece_new[2][kWarps], piece_old[2][kWarps];
  uint64_t prev_tot[4];            // narrow jobs: {cnt, R, G, B} sums of the previous pass (fixed-point detection)
  int32_t converged;
  int32_t n_nodes, n_prev, njobs, prev_njobs;
  int32_t nwide_tiles, n_mywide, n_mynarrow;
  int32_t mode;  // 0 = threshold policy, 1 = replicated sequential replay
  int32_t done, bad;
  int32_t new_index, old_index;
  int32_t scan_carry;
  int32_t warp_tmp[32];
  uint32_t cur_old, cur_new;
  uint32_t num_points;
  tie::PassExt ext;   // tie audit: centres and bounds behind S.pp (written with it)
  JobAudit aud;       // tie audit: constants of the narrow job in flight
  JobAudit wide_aud[kAudCache];
  uint32_t near;     // tie audit: points of the pass just reduced / gathered that sit inside the noise bound
  uint32_t job_tie;   // TieBit mask of the narrow job in flight
  uint32_t tie_total; // TieBit mask of the frame (CTA 0, final assignment + palette)
  uint32_t cut_count; // consumed splits whose cut is flagged (kTieCut): entries of the second list of SplitArgs::tie_list
  CutOverride ovr[kCutOverrideCap];  // SplitArgs::cut_overrides, staged
  uint32_t n_ovr;
  NarrowGroup grp[kGroups];
  int32_t narrow_next;  // entries of mynarrow handed to the groups so far
};

// Barriers of the helpers that run either on the whole CTA or on one narrow-job group (named barrier 1 + group).
struct CtaSync {
  __device__ __forceinline__ void operator()() const { __syncthreads(); }
};
struct GroupSync {
  int id;
  __device__ __forceinline__ void operator()() const { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(kGroupT) : "memory"); }
};

struct Arrays {
  double *tse;         // [cap]
  int32_t *child;      // [cap]
  uint32_t *size;      // [cap]
  int32_t *parent;     // [cap]
  int32_t *jobnode;    // [K]
  uint32_t *tile0;     // [K+1] wide-tile prefix
  uint32_t *slot0;     // [K+1] slot prefix
  uint32_t *nidx;      // [K+1] narrow ordinal prefix
  uint16_t *mywide;    // [K]
  uint16_t *mynarrow;  // [K]
  int32_t *cnode;      // [K]   cluster -> node (final assignment / sequential replay)
  double *ctse;        // [K]
  int32_t *cand;       // [K]
  int32_t *rank;       // [cap]  number of known nodes with a larger TSE (final assignment)
  double *terr;        // [cap]  tie audit: bound of the node's TSE
  int32_t *byrank;     // [cap]  tie audit: node of every TSE rank (final assignment)
  uint8_t *jobtie;     // [K]    tie audit: TieBit mask of this round's wide jobs (owner CTA)
  // Fixed-point exit of this CTA's wide jobs, indexed like mywide.  Only the controller's selection uses rank[] and cand[],
  // so these two live in their memory.
  uint64_t (*wprev)[4];  // [K]  {cnt, R, G, B} of the last pass gathered (in rank[], cap * 4 >= K * 32 bytes)
  int32_t *wfin;         // [K]  1 + the pass that ran as the job's final one, 0 while it runs (in cand[])
  // [Split2Extra::wide_cache_points] this CTA's shares of the round's wide jobs, back to back in mywide order, as far as they
  // fit: written by the cut pass, read by the later passes and the partition of the same round
  uint2 *wcache;
};

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long *p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_relaxed_u32(const unsigned int *p) {
  unsigned int v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Every wait on another CTA is bounded: a persistent spinning kernel must never be able to wedge the
// device.  After kSpinCycles without progress the waiter records where it was stuck in ctl[] and
// raises ctl[kCtlError]; every other waiter sees the flag and leaves too, and the host reports it.
constexpr long long kSpinCycles = 400000000ll;  // default: ~0.2 s at 1.9 GHz; a healthy wait is microseconds
// (SplitArgs::spin_cycles, DIVQUANT_B200_SPIN_MS, replaces it: compute-sanitizer, cuda-gdb or heavy time-slicing can make a
// healthy wait long)

__device__ __forceinline__ bool spin_expired(const SplitArgs &A, long long t0, unsigned &polls, int what, int arg) {
  if ((++polls & 1023u) != 0) return false;
  if (ld_relaxed_u32(A.ctl + kCtlError) != 0) return true;
  if (clock64() - t0 > (A.spin_cycles > 0 ? A.spin_cycles : kSpinCycles)) {
    if (atomicCAS(A.ctl + kCtlError, 0u, 3u) == 0u) {
      A.ctl[kCtlWords - 1] = (uint32_t)what;
      A.ctl[kCtlJobs] = (uint32_t)arg;
      A.ctl[kCtlTiles] = blockIdx.x;
      A.ctl[kCtlNodes] = ld_relaxed_u32(A.barrier);
    }
    return true;
  }
  return false;
}

#define DQ_PROGRESS(code) \
  do {                     \
    if (threadIdx.x == 0) X.progress[blockIdx.x] = (uint32_t)(code); \
  } while (0)

// CTA-uniform view of the error flag.
__device__ __forceinline__ bool cta_error(const SplitArgs &A, Shared2 &S) {
  __syncthreads();
  if (threadIdx.x == 0) S.bad = (int32_t)ld_relaxed_u32(A.ctl + kCtlError);
  __syncthreads();
  const bool e = S.bad != 0;
  __syncthreads();
  return e;
}

// Grid barrier: relaxed polling (no L1 invalidation per poll), one fence on each side.
__device__ __forceinline__ void grid_barrier2(const SplitArgs &A, unsigned int &target, uint32_t *progress = nullptr) {
  unsigned int *counter = A.barrier;
  __syncthreads();
  if (threadIdx.x == 0) {
    target += gridDim.x;
    if (progress) progress[blockIdx.x] = 900000u + target;
    __threadfence();
    atomicAdd(counter, 1u);
    const long long t0 = clock64();
    unsigned polls = 0;
    while (ld_relaxed_u32(counter) < target) {
      if (spin_expired(A, t0, polls, 1, (int)target)) break;
    }
    __threadfence();
  }
  __syncthreads();
}

#include "dq_split_ordered.cuh"

__device__ __forceinline__ void trace2(const SplitArgs &A, int tag, int arg) {
  if (A.timeline != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
    const unsigned long long n = A.timeline[0];
    if (2 * n + 3 < A.timeline_cap) {
      A.timeline[1 + 2 * n] = ((unsigned long long)tag << 32) | (unsigned)arg;
      A.timeline[2 + 2 * n] = clock64();
      A.timeline[0] = n + 1;
    }
  }
}

// ---- block-level helpers ----------------------------------------------------------------------------

// Warp sum of values below 2^50 with the REDUX unit (2 cycles per REDUX per SM, against ten dependent
// shuffles for a 64-bit butterfly): one 32-bit REDUX when every lane is below 2^27 (warp-uniform
// branch), otherwise two 24/26-bit limbs.
__device__ __forceinline__ uint64_t warp_sum_redux(uint64_t v) {
  if (!__any_sync(0xffffffffu, (v >> 27) != 0)) return __reduce_add_sync(0xffffffffu, (unsigned)v);
  const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)(v & 0xFFFFFFu));
  const unsigned hi = __reduce_add_sync(0xffffffffu, (unsigned)(v >> 24));
  return (uint64_t)lo + ((uint64_t)hi << 24);
}

// Stage 1 of a CTA-wide sum: the first `warps` warps reduce their WORDS values into S.red[warp][].
// One vote decides for all words whether a single 32-bit REDUX per word is enough (every lane below 2^27,
// the usual case) or two 24/26-bit limbs are needed: the REDUX unit, not latency, bounds this stage
// (tools/microbench/classify_mb.cu: 340 cycles against 500 with a vote per word and 1000 with two limbs always).
// Ends with a barrier.
template <int WORDS, typename St, typename Sync = CtaSync>
__device__ __forceinline__ void reduce_stage1(St &S, const uint64_t (&v)[kAccWords], int warps, int t = threadIdx.x, Sync sync = Sync()) {
  const int lane = t & 31, warp = t >> 5;
  if (warp < warps) {
    uint64_t all = 0;
#pragma unroll
    for (int w = 0; w < WORDS; ++w) all |= v[w];
    uint64_t s[WORDS];
    if (!__any_sync(0xffffffffu, (all >> 27) != 0)) {
#pragma unroll
      for (int w = 0; w < WORDS; ++w) s[w] = __reduce_add_sync(0xffffffffu, (unsigned)v[w]);
    } else {
#pragma unroll
      for (int w = 0; w < WORDS; ++w) {
        const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)(v[w] & 0xFFFFFFu));
        const unsigned hi = __reduce_add_sync(0xffffffffu, (unsigned)(v[w] >> 24));
        s[w] = (uint64_t)lo + ((uint64_t)hi << 24);
      }
    }
    if (lane == 0) {
#pragma unroll
      for (int w = 0; w < WORDS; ++w) S.red[warp][w] = s[w];
    }
  }
  sync();
}

// Stage 2, executed by warp 0 only: sums rows 0..rows-1 (<= 32) of S.red (values below 2^54) into
// S.tot with two 27-bit limbs per word.  Totals are visible to warp 0 on return (no CTA barrier).
template <int WORDS, typename St>
__device__ __forceinline__ void reduce_stage2_warp0(St &S, int rows) {
  const int lane = threadIdx.x & 31;
  uint64_t x[WORDS];
#pragma unroll
  for (int w = 0; w < WORDS; ++w) x[w] = lane < rows ? S.red[lane][w] : 0ull;
#pragma unroll
  for (int w = 0; w < WORDS; ++w) {
    const unsigned a = __reduce_add_sync(0xffffffffu, (unsigned)(x[w] & 0x7FFFFFFu));
    const unsigned c = __reduce_add_sync(0xffffffffu, (unsigned)(x[w] >> 27));
    if (lane == 0) S.tot[w] = (uint64_t)a + ((uint64_t)c << 27);
  }
  __syncwarp();
}

// Tie audit: the classification adds (near ? 1 : 0) << 32 per thread to the point counter (kAccPts), so the number of
// threads that saw a point inside the noise bound rides through every reduction and exchange for free.  Warp 0 calls
// this once the totals are in S.tot: S.near = that number, S.tot[kAccPts] = the plain point count again.
template <typename St>
__device__ __forceinline__ void split_near_warp0(St &S, int t = threadIdx.x) {
  if (t == 0) {
    S.near = (uint32_t)(S.tot[kAccPts] >> 32);
    S.tot[kAccPts] &= 0xFFFFFFFFull;
  }
  __syncwarp();
}

// Sum of v[0..WORDS) over the first `warps` warps of the CTA into S.tot, visible to all threads.
template <int WORDS>
__device__ __forceinline__ void block_total(Shared2 &S, const uint64_t (&v)[kAccWords], int warps = kWarps) {
  reduce_stage1<WORDS>(S, v, warps);
  if (threadIdx.x < 32) reduce_stage2_warp0<WORDS>(S, warps);
  __syncthreads();
}

// In-place exclusive scan of a[0..n) in shared memory; total left in S.scan_carry.
__device__ void block_scan(Shared2 &S, uint32_t *a, int n) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (n + T - 1) / T;
  const int lo = min(tid * per, n), hi = min(lo + per, n);
  uint32_t sum = 0;
  for (int i = lo; i < hi; ++i) sum += a[i];
  uint32_t incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) S.warp_tmp[warp] = (int32_t)incl;
  __syncthreads();
  if (warp == 0) {
    const uint32_t w = lane < kWarps ? (uint32_t)S.warp_tmp[lane] : 0u;
    uint32_t wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += t;
    }
    S.warp_tmp[lane] = (int32_t)(wi - w);
    if (lane == 31) S.scan_carry = (int32_t)wi;
  }
  __syncthreads();
  uint32_t run = (uint32_t)S.warp_tmp[warp] + (incl - sum);
  for (int i = lo; i < hi; ++i) {
    const uint32_t t = a[i];
    a[i] = run;
    run += t;
  }
  __syncthreads();
}

// Appends, in ascending order, every i in [lo, hi) with pred(i) to out[*count..]; all threads call.
template <typename Pred, typename Out>
__device__ void ordered_compact(Shared2 &S, int lo, int hi, Pred pred, Out out, int32_t *count) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int base = lo; base < hi; base += T) {
    const int i = base + tid;
    const bool p = (i < hi) && pred(i);
    const unsigned ballot = __ballot_sync(0xffffffffu, p);
    if (lane == 0) S.warp_tmp[warp] = __popc(ballot);
    __syncthreads();
    // every warp scans the 32 warp counts itself (one shuffle ladder, no extra barrier)
    const int mine = lane < kWarps ? S.warp_tmp[lane] : 0;
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    const int before = *count + __shfl_sync(0xffffffffu, incl - mine, warp);
    if (p) out(before + __popc(ballot & ((1u << lane) - 1u)), i);
    __syncthreads();
    if (tid == 0) *count += total;
    __syncthreads();
  }
}

__device__ __forceinline__ SplitNode load_node(const SplitArgs &A, const Shared2 &S, int id) {
  if (id == 0) return S.root;
  SplitNode nd;
  const double *src = reinterpret_cast<const double *>(A.nodes + id);
  double *dst = reinterpret_cast<double *>(&nd);
#pragma unroll
  for (int i = 0; i < (int)(sizeof(SplitNode) / 8); ++i) dst[i] = __ldcg(src + i);
  return nd;
}

// Classification parameters of the next pass from the totals in S.tot, computed by warp 0
// (one lane per channel), left in S.pp.  Caller synchronises afterwards.
template <typename St>
__device__ __forceinline__ void derive_params_warp0(St &S, const JobConst &jc, double norm, int t = threadIdx.x) {
  if (t < 32) {  // uniform per warp
    const int c = min(t, 2);
    const double nw = fmul(u52_to_double(S.tot[kAccCnt]), norm);
    const double nm = fdiv(fmul(u52_to_double(S.tot[kAccR + c]), norm), nw);
    const double ow = fsub(jc.tw, nw);
    const double om = fdiv(fsub(fmul(jc.tw, jc.tm[c]), fmul(nw, nm)), ow);
    const double a = fsq(om), b = fsq(nm);
    const double a1 = __shfl_sync(0xffffffffu, a, 1), b1 = __shfl_sync(0xffffffffu, b, 1);
    const double a2 = __shfl_sync(0xffffffffu, a, 2), b2 = __shfl_sync(0xffffffffu, b, 2);
    if (t < 3) {
      S.pp.r[c] = fsub(om, nm);
      S.ext.om[c] = om;  // (tie audit: the centres themselves, for the cold per-point re-check)
      S.ext.nm[c] = nm;
    }
    if (t == 0) {
      double l = fsub(a, b);  // (:616-619), left to right
      l = fadd(l, a1);
      l = fsub(l, b1);
      l = fadd(l, a2);
      l = fsub(l, b2);
      S.pp.a = fmul(0.5, l);
      S.pp.axis = jc.axis;
      S.pp.buf = jc.buf;
      S.pp.begin = jc.begin;
      S.pp.size = jc.size;
    }
  }
}

// Tie audit, next to derive_params_warp0 and at the same time: WARP 1 sums the rows of S.red itself (the totals warp 0
// is reducing into S.tot), derives the same centres and from them the tolerance of the next pass's hyperplane test
// (dq_tie.cuh), so that the bound costs the split's critical path nothing.  Writes S.pp.tol_hi and S.ext only.
template <typename St>
__device__ __forceinline__ uint64_t warp_total_row(const St &S, int lane, int rows, int w) {
  const uint64_t x = lane < rows ? S.red[lane][w] : 0ull;
  const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)(x & 0x7FFFFFFu));
  const unsigned hi = __reduce_add_sync(0xffffffffu, (unsigned)(x >> 27));
  return (uint64_t)lo + ((uint64_t)hi << 27);
}
template <typename St>
__device__ __forceinline__ void derive_audit_warp1(St &S, const JobConst &jc, const JobAudit *aud, double norm, int rows,
                                                   int t = threadIdx.x) {
  if (t >= 32 && t < 64) {  // uniform per warp
    const int lane = t & 31;
    const double eM = aud ? aud->eM : 0.0;
    if (eM < 0.0) {  // audit off
      if (lane == 0) S.pp.tol_hi = -1;
      return;
    }
    if (aud == nullptr) {  // beyond the cache: every point counts as inside the noise (never seen in practice)
      if (lane == 0) {
        S.ext.tol = __longlong_as_double(0x7ff0000000000000ll);
        S.ext.e_om = S.ext.e_nm = S.ext.tol;
        S.pp.tol_hi = 0x7ff00001;
      }
      return;
    }
    // Only the new side's weight and point count are needed: the centres' magnitudes enter the bounds as 256 (they are
    // means of bytes), so no division happens here and this warp is never the one the pass waits for.
    const uint64_t t_cnt = warp_total_row(S, lane, rows, kAccCnt), t_pts = warp_total_row(S, lane, rows, kAccPts);
    const double nw = fmul(u52_to_double(t_cnt), norm);
    const double ow = fsub(jc.tw, nw);
    if (lane == 0) {
      const tie::PassErr q = tie::pass_err_fast(aud->eW, aud->eS, jc.tw, aud->m1, nw, 256.0, ow, 256.0, (double)(uint32_t)t_pts);
      const double tol = tie::hyperplane_tol(q);
      S.ext.e_om = q.e_om;
      S.ext.e_nm = q.e_nm;
      S.ext.tol = tol;
      S.pp.tol_hi = __double2hiint(tol) + (tol >= 0.0 ? 1 : 0);
    }
  }
}

template <typename St>
__device__ __forceinline__ void set_split_params(const Shared2 &S, St &G, const JobConst &jc, const JobAudit *aud,
                                                 int t = threadIdx.x) {
  if (t == 0) {
    G.pp.a = jc.cut;
    // a cut taken from SplitArgs::cut_overrides is the reference's own comparison: not audited
    bool forced = false;
    for (uint32_t i = 0; i < S.n_ovr; ++i)
      forced = forced || (S.ovr[i].begin == jc.begin && S.ovr[i].size == jc.size && S.ovr[i].mean_ref == jc.cut);
    const double eM = forced ? -1.0 : (aud ? aud->eM : __longlong_as_double(0x7ff0000000000000ll));
    G.ext.tol = eM;  // tie audit of the cut test (:473): the cut is the node's mean (a forced cut is the reference's own)
    G.pp.tol_hi = __double2hiint(eM) + (eM >= 0.0 ? 1 : 0);
    G.pp.r[0] = G.pp.r[1] = G.pp.r[2] = 0.0;
    G.pp.axis = jc.axis;
    G.pp.buf = jc.buf;
    G.pp.begin = jc.begin;
    G.pp.size = jc.size;
  }
}

__device__ __forceinline__ JobAudit job_audit_of(const SplitNode &nd, bool audit) {
  JobAudit a;
  a.eW = nd.eW;
  a.eS = nd.eS;
  a.m1 = tie::max3abs(nd.tm);
  a.eM = audit ? nd.eM : -1.0;
  return a;
}
__device__ __forceinline__ JobConst job_const_of(const SplitNode &nd) {
  JobConst jc;
  jc.tw = nd.tw;
  jc.tm[0] = nd.tm[0], jc.tm[1] = nd.tm[1], jc.tm[2] = nd.tm[2];
  choose_cut(nd.tv, nd.tm, jc.axis, jc.cut);
  jc.buf = nd.buf;
  jc.begin = nd.begin;
  jc.size = nd.size;
  return jc;
}
__device__ __forceinline__ JobConst job_const_of(const Shared2 &S, const SplitNode &nd) {
  JobConst jc = job_const_of(nd);
  for (uint32_t i = 0; i < S.n_ovr; ++i) {
    if (S.ovr[i].begin == jc.begin && S.ovr[i].size == jc.size && S.ovr[i].mean_here == jc.cut) {
      jc.cut = S.ovr[i].mean_ref;
    }
  }
  return jc;
}

__device__ __forceinline__ void add_point(uint64_t (&v)[kAccWords], uint2 p, bool with_squares) {
  const uint64_t cnt = p.y, R = (p.x >> 16) & 0xFFu, G = (p.x >> 8) & 0xFFu, B = p.x & 0xFFu;
  v[kAccCnt] += cnt;
  v[kAccR] += cnt * R;
  v[kAccG] += cnt * G;
  v[kAccB] += cnt * B;
  v[kAccPts] += 1;
  if (with_squares) {
    v[kAccRR] += cnt * (R * R);
    v[kAccGG] += cnt * (G * G);
    v[kAccBB] += cnt * (B * B);
  }
}

// Owner of a finished split writes its two children (totals of the last pass in S.tot, parent in S.cur).
template <typename St>
__device__ __forceinline__ void write_children(const SplitArgs &A, St &S, int node_id, int child0, const JobConst &jc,
                                               uint32_t tie_bits, int t = threadIdx.x) {
  if (t == 0) {
    SplitNode o, n;
    make_children(S.cur, node_id, child0, A.norm, S.tot, o, n, A.tie_audit != 0u);
    A.nodes[child0] = o;
    A.nodes[child0 + 1] = n;
    SplitNode *p = A.nodes + node_id;
    p->child = child0;
    p->axis = jc.axis;
    p->cut = jc.cut;
    p->tie = tie_bits;  // decisions of this split inside the reference's noise (counted if the split is consumed)
  }
}

// ---- exchange of partial sums between the CTAs of a wide job ------------------------------------------

template <int WORDS>
__device__ __forceinline__ void publish(unsigned long long *slots, uint32_t slot, const Shared2 &S, unsigned tag) {
  if (threadIdx.x < WORDS)
    st_relaxed_u64(slots + (size_t)slot * kAccWords + threadIdx.x, ((unsigned long long)tag << 48) | S.tot[threadIdx.x]);
}

// Waits for the m participants' words of this pass and leaves their sums in S.tot.
__device__ __forceinline__ void gather(const SplitArgs &A, Shared2 &S, const unsigned long long *slots, uint32_t slot0,
                                       int m, int words, unsigned tag) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int w = tid & 7;
  unsigned long long sum = 0;
  if (w < words) {
    for (int i = tid >> 3; i < m; i += T / 8) {
      const unsigned long long *p = slots + (size_t)(slot0 + i) * kAccWords + w;
      unsigned long long v;
      const long long t0 = clock64();
      unsigned polls = 0;
      do {
        v = ld_relaxed_u64(p);
      } while ((unsigned)(v >> 48) != tag && !spin_expired(A, t0, polls, 2, (int)((tag << 16) | (unsigned)i)));
      sum += v & kValueMask;
    }
  }
  sum += __shfl_xor_sync(0xffffffffu, sum, 8);
  sum += __shfl_xor_sync(0xffffffffu, sum, 16);
  if (lane < 8) S.red[warp][lane] = sum;
  __syncthreads();
  if (tid < 32) {
    reduce_stage2_warp0<kAccWords>(S, kWarps);
    split_near_warp0(S);
  }
  // no barrier here: callers let warp 0 go on (parameter derivation) and synchronise afterwards
}

// Results to the host mailbox (see SplitArgs::mailbox).  Called by every thread of CTA 0 after the palette is in place.
__device__ __forceinline__ void publish_mailbox(const SplitArgs &A, uint32_t U) {
  if (A.mailbox == nullptr) return;
  __syncthreads();  // palette / result / ctl written by this CTA are visible to it
  volatile uint32_t *mb = A.mailbox;
  const int tid = threadIdx.x, K = (int)A.num_colors;
  for (int i = tid; i < K; i += T) mb[kMailboxPalette + i] = A.palette[i];
  if (tid < 4) mb[2 + tid] = A.result[tid];
  if (tid < (int)kCtlWords) mb[6 + tid] = A.ctl[tid];
  if (tid == 0) mb[1] = U;
  __threadfence_system();
  __syncthreads();
  if (tid == 0) mb[0] = A.mailbox_seq;
}

// ---- final assignment of cluster indices --------------------------------------------------------------

// Palette = rounded means of the non-empty clusters in index order (:1030-1065). cnode[ic] = node of cluster ic.
__device__ void emit_palette(const SplitArgs &A, Shared2 &S, const Arrays &R) {
  const int tid = threadIdx.x, lane = tid & 31, K = (int)A.num_colors;
  if (tid == 0) {
    S.scan_carry = 0;
    S.cur_new = 0u;  // (free here) number of clusters whose rounding is flagged
  }
  __syncthreads();
  for (int base = 0; base < K; base += T) {
    const int ic = base + tid;
    uint32_t colour = 0, size = 0;
    bool flagged = false;
    if (ic < K) {
      double mean[3] = {0.0, 0.0, 0.0};  // K == 1 never assigns mean[0] (SURVEY 7 quirk)
      if (K > 1) {
        const SplitNode nd = load_node(A, S, R.cnode[ic]);
        size = nd.size;
        mean[0] = nd.tm[0], mean[1] = nd.tm[1], mean[2] = nd.tm[2];
        if (A.tie_audit != 0u && size > 0 &&
            (tie::round_tie(mean[0], nd.eM) || tie::round_tie(mean[1], nd.eM) || tie::round_tie(mean[2], nd.eM))) {
          atomicOr(&S.tie_total, (uint32_t)kTieRound);  // D5 (:1050-1052)
          flagged = true;
        }
      } else {
        size = S.num_points;
      }
      if (size > 0) {
        const uint32_t Rr = (__double2uint_rz(fadd(mean[0], 0.5)) & 0xFFu) << A.shift;
        const uint32_t Gg = (__double2uint_rz(fadd(mean[1], 0.5)) & 0xFFu) << A.shift;
        const uint32_t Bb = (__double2uint_rz(fadd(mean[2], 0.5)) & 0xFFu) << A.shift;
        colour = (Rr << 16) | (Gg << 8) | Bb;
      }
      A.cluster_size[ic] = size;
      A.cluster_mean[3 * ic + 0] = mean[0];
      A.cluster_mean[3 * ic + 1] = mean[1];
      A.cluster_mean[3 * ic + 2] = mean[2];
    }
    const unsigned ballot = __ballot_sync(0xffffffffu, size > 0);
    if (lane == 0) S.warp_tmp[tid >> 5] = __popc(ballot);
    __syncthreads();
    int before = S.scan_carry;
    for (int w = 0; w < (tid >> 5); ++w) before += S.warp_tmp[w];
    if (size > 0) A.palette[before + __popc(ballot & ((1u << lane) - 1u))] = colour;
    if (flagged && A.tie_list != nullptr) {  // for dq_resolve.cu: which cluster, which node, which palette word
      const uint32_t at = atomicAdd(&S.cur_new, 1u);
      if (at < kTieListCap) {
        uint32_t *e = A.tie_list + 4 * at;
        e[0] = (uint32_t)ic;
        e[1] = (uint32_t)R.cnode[ic];
        e[2] = (uint32_t)(before + __popc(ballot & ((1u << lane) - 1u)));
        e[3] = 0u;
      }
    }
    __syncthreads();
    if (tid == 0) {
      int tot = 0;
      for (int w = 0; w < kWarps; ++w) tot += S.warp_tmp[w];
      S.scan_carry += tot;
    }
    __syncthreads();
  }
  if (tid == 0) {
    A.result[0] = (uint32_t)S.scan_carry;
    A.result[1] = (uint32_t)(K - S.scan_carry);
    A.ctl[kCtlTieCount] = S.cur_new;
    A.ctl[kCtlCutCount] = (A.tie_audit != 0u && S.mode == 0) ? S.cut_count : 0u;
  }
}

__device__ void write_record(const SplitArgs &A, const Shared2 &S, int node, int child, int new_index, int old_index) {
  // the parent comes from global memory even for the root: its owner stored axis/cut there
  const SplitNode p = A.nodes[node], o = load_node(A, S, child), n = load_node(A, S, child + 1);
  SplitRecord r;
  r.new_index = new_index;
  r.old_index = old_index;
  r.cut_axis = p.axis;
  r.num_points = (int32_t)p.size;
  r.new_size = (int32_t)n.size;
  r.is_last = (new_index == (int)A.num_colors - 1);
  r.cut_pos = p.cut;
  r.total_weight = p.tw;
  r.new_weight = n.tw;
  r.old_weight = o.tw;
  for (int c = 0; c < 3; ++c) {
    r.new_mean[c] = n.tm[c];
    r.old_mean[c] = o.tm[c];
    r.new_var[c] = n.tv[c];
    r.old_var[c] = o.tv[c];
  }
  r.new_tse = n.tse;
  r.old_tse = o.tse;
  A.records[new_index - 1] = r;
}

// Parallel reconstruction of the reference's sequence when the TSE order is strict.
//
// With key(root) = +inf: the nodes the reference pops are L = the K-1 known nodes of largest TSE, in
// descending TSE order, PROVIDED every one of them is a computed split, has a TSE above DBL_MIN, is
// strictly below its parent (so the parent is popped first) and no two compared values are equal
// (ties are resolved by cluster index in the reference, :882).  All of that is checked; on any doubt
// S.bad is set and the caller falls back to the sequential scan.  On success R.cnode[ic] = node of
// final cluster ic: the split popped at step t creates cluster t from its "new" child, the "old"
// child inherits the parent's index.
__device__ void fast_assignment(const SplitArgs &A, Shared2 &S, const Arrays &R) {
  const int tid = threadIdx.x, K = (int)A.num_colors, n = S.n_nodes;
  if (tid == 0) {
    S.bad = 0;
    S.scan_carry = 0;  // |L|
  }
  for (int i = tid; i < (K + 31) / 32; i += T) R.cand[i] = 0;  // bitmap of popped ranks
  __syncthreads();
  // rank[i] = number of known nodes with a larger TSE
  const bool audit = A.tie_audit != 0u;
  for (int i = tid; i < n; i += T) {
    const double t = R.tse[i];
    int above = n;
    if (t == t) {  // NaN is never selected (:882)
      above = 0;
#pragma unroll 8
      for (int m2 = 0; m2 < n; ++m2) above += (R.tse[m2] > t);
    }
    R.rank[i] = above;
  }
  __syncthreads();
  uint32_t near_mask = 0u;  // per thread: bit q = its q-th node may have another node's TSE within the two bounds
  if (audit) {
    // tie audit, D4, for the nodes the reference pops: does any other node's TSE come within the two bounds of this one?
    // The ranks just computed ARE the descending TSE order, so only a node's neighbours in that order can be that close:
    // byrank[] inverts the ranks (equal TSEs share a rank and collide there: a tie by definition), and a node is marked
    // when a neighbour lies within its own bound plus the LARGEST bound of any node -- a superset of the exact pairwise
    // test, which follows below for the few nodes marked here (together with whether the other node matters at all).
    for (int i = tid; i < n; i += T) R.byrank[i] = -1;
    __shared__ double s_emax;
    if (tid == 0) s_emax = 0.0, S.cut_count = 0u;
    __syncthreads();
    double emax = 0.0;
    for (int i = tid; i < n; i += T) {
      const int r = R.rank[i];
      if (r < n) R.byrank[r] = i;
      const double e = R.terr[i];
      if (e > emax || e != e) emax = (e != e) ? __longlong_as_double(0x7ff0000000000000ll) : e;
    }
    if (emax > 0.0) atomicMax(reinterpret_cast<unsigned long long *>(&s_emax), (unsigned long long)__double_as_longlong(emax));
    __syncthreads();
    emax = s_emax;
    int q = 0;
    for (int i = tid; i < n; i += T, ++q) {
      const int r = R.rank[i];
      if (r >= K - 1 || i == 0) continue;
      const double t = R.tse[i], tol = R.terr[i] + emax;
      bool near = R.byrank[r] != i;  // somebody with an equal TSE took the slot
      for (int d = r - 1; d >= 0 && !near; --d) {  // next node above (slots emptied by equal TSEs are skipped)
        const int j = R.byrank[d];
        if (j < 0) continue;
        near = fabs(R.tse[j] - t) <= tol;
        break;
      }
      for (int d = r + 1; d < n && !near; ++d) {  // next node below
        const int j = R.byrank[d];
        if (j < 0) continue;
        near = fabs(R.tse[j] - t) <= tol;
        break;
      }
      if (near) near_mask |= 1u << (q & 31);
    }
  }
  for (int i = tid; i < n; i += T) {
    const double t = R.tse[i];
    const int above = R.rank[i];
    if (above < K - 1) {
      atomicAdd(&S.scan_carry, 1);
      bool ok = (R.child[i] >= 0) && (t > DBL_MIN);
      if (i != 0) ok = ok && (R.tse[R.parent[i]] > t);
      // equal keys share a rank: every popped rank 0..K-2 must be hit exactly once (checked through |L| == K-1
      // together with the bitmap below), and nothing may tie with the first rejected key
      if (ok) {
        const unsigned bit = 1u << (above & 31);
        if (atomicOr(reinterpret_cast<unsigned *>(R.cand) + (above >> 5), bit) & bit) ok = false;
      }
      if (!ok) S.bad = 1;
    }
  }
  __syncthreads();
  if (S.scan_carry != K - 1 && tid == 0) S.bad = 1;
  __syncthreads();
  if (S.bad) return;
  if (A.tie_audit != 0u) {
    // D4 (:876-887): the reference pops the same nodes in the same order if every popped node's TSE is separated from the
    // DBL_MIN seed and from the TSE of every other node of the reference's sequence (popped nodes and their children) by
    // more than the two bounds.  Also collects the decisions flagged inside the consumed splits themselves.
    uint32_t bits = 0u;
    int q = 0;
    for (int i = tid; i < n; i += T, ++q) {
      if (R.rank[i] >= K - 1) continue;
      const uint32_t node_bits = __ldcg(&A.nodes[i].tie);
      bits |= node_bits;
      if ((node_bits & (uint32_t)kTieCut) && A.tie_list != nullptr) {  // for dq_resolve.cu: whose mean decides the cut
        const uint32_t at = atomicAdd(&S.cut_count, 1u);
        if (at < kTieListCap && blockIdx.x == 0) A.tie_list[kTieCutList + at] = (uint32_t)i;
      }
      if (i == 0) continue;  // the root is split first, unconditionally
      const double t = R.tse[i], e = R.terr[i];
      if (!(t - e > DBL_MIN)) bits |= (uint32_t)kTieTse;
      if (!((near_mask >> (q & 31)) & 1u) && q < 32) continue;
      for (int m2 = 1; m2 < n; ++m2) {
        if (m2 == i) continue;
        const bool relevant = R.rank[m2] < K - 1 || R.rank[R.parent[m2]] < K - 1;
        if (relevant && fabs(R.tse[m2] - t) <= e + R.terr[m2]) bits |= (uint32_t)kTieTse;
      }
    }
    if (bits) atomicOr(&S.tie_total, bits);
  }
  for (int i = tid; i < n; i += T) {
    const bool popped = R.rank[i] < K - 1;
    const bool final_cluster = !popped && i != 0 && R.rank[R.parent[i]] < K - 1;
    if (!popped && !final_cluster) continue;
    // cluster index carried by node i: up the chain of "old" children to the nearest "new" child
    int cur = i, idx = 0;
    while (cur != 0) {
      const int p = R.parent[cur];
      if (cur == R.child[p] + 1) {
        idx = R.rank[p] + 1;
        break;
      }
      cur = p;
    }
    if (popped) {
      if (A.records != nullptr && blockIdx.x == 0) write_record(A, S, i, R.child[i], R.rank[i] + 1, idx);
    } else {
      R.cnode[idx] = i;
    }
  }
  __syncthreads();
}

// The reference's sequential selection (:876-887) over the cached splits, replicated in every CTA.
// Leaves S.done = 1 when all K-1 splits were consumed; otherwise fills the job list with the stalled
// split plus the leaves inside the remaining budget (ordered by cluster index).
__device__ void sequential_controller(const SplitArgs &A, Shared2 &S, const Arrays &R) {
  const int tid = threadIdx.x, lane = tid & 31, K = (int)A.num_colors;
  if (tid < 32) {
    int new_index = S.new_index, old_index = S.old_index;
    while (new_index < K) {
      const int node = R.cnode[old_index];
      const int child = R.child[node];
      if (child < 0) break;
      __syncwarp();
      if (lane == 0) {
        R.cnode[old_index] = child;
        R.cnode[new_index] = child + 1;
        if (A.records != nullptr && blockIdx.x == 0) write_record(A, S, node, child, new_index, old_index);
      }
      if (new_index == K - 1) {
        new_index = K;
        break;
      }
      if (lane == 0) {
        R.ctse[old_index] = R.tse[child];
        R.ctse[new_index] = R.tse[child + 1];
      }
      __syncwarp();
      double best = DBL_MIN;
      int best_i = -1;
      for (int ic = lane; ic <= new_index; ic += 32) {
        const double t = R.ctse[ic];
        if (best < t) {
          best = t;
          best_i = ic;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
        const bool take = (oi >= 0) && (best_i < 0 || best < ob || (ob == best && oi < best_i));
        if (take) {
          best = ob;
          best_i = oi;
        }
      }
      if (best_i >= 0) old_index = best_i;
      ++new_index;
    }
    if (lane == 0) {
      S.new_index = new_index;
      S.old_index = old_index;
    }
  }
  __syncthreads();
  const int new_index = S.new_index, old_index = S.old_index;
  if (new_index >= K) {
    if (tid == 0) {
      S.done = 1;
      S.njobs = 0;
    }
    __syncthreads();
    return;
  }
  // requests: the stalled cluster + the top-(R-1) other unsplit clusters by (tse desc, index asc)
  const int budget = (K - new_index) - 1;
  if (tid == 0) {
    S.njobs = 0;
    S.scan_carry = 0;
  }
  __syncthreads();
  int32_t *ncand = &S.scan_carry;
  // candidates in cluster-index order
  ordered_compact(
      S, 0, new_index,
      [&](int ic) { return ic != old_index && R.child[R.cnode[ic]] < 0 && (R.ctse[ic] > DBL_MIN); },
      [&](int pos, int ic) { R.cand[pos] = ic; }, ncand);
  const int nc = *ncand;
  __syncthreads();
  // mark the clusters to split: flag = -(ic+1) stays, others removed
  for (int i = tid; i < nc; i += T) {
    const int ic = R.cand[i];
    bool take = true;
    if (nc > budget) {
      const double mine = R.ctse[ic];
      int rank = 0;
      for (int q = 0; q < nc; ++q) {
        const int oc = R.cand[q];
        const double t = R.ctse[oc];
        rank += (t > mine) || (t == mine && oc < ic);
      }
      take = rank < budget;
    }
    R.cand[i] = take ? ic : -1;
  }
  __syncthreads();
  if (tid == 0) {
    R.jobnode[0] = R.cnode[old_index];  // the stalled split first
    S.njobs = 1;
  }
  __syncthreads();
  ordered_compact(
      S, 0, nc, [&](int i) { return R.cand[i] >= 0; }, [&](int pos, int i) { R.jobnode[pos] = R.cnode[R.cand[i]]; },
      &S.njobs);
  __syncthreads();
}

// One pass of a narrow job: classify the (register-resident) points, reduce, and -- except after the
// last pass -- derive the next pass's parameters.  SPLIT: cut test of pass 0; FINAL: last LKM pass
// (also sums count*c*c).  Returns the membership mask of this thread's points.
template <bool SPLIT, bool FINAL, typename St, typename Sync>
__device__ __forceinline__ unsigned narrow_pass(St &S, const uint2 (&p)[kNarrowPPT], unsigned validmask, int ppt, int nwarps,
                                                const JobConst &jc, double norm, int t, Sync sync) {
  // (tie audit constants of the narrow job in flight: S.aud)
  const PassParams pp = S.pp;
  AccD acc = acc_zero();
  unsigned newmask = 0;
  bool near = false;
#pragma unroll
  for (int k = 0; k < kNarrowPPT; ++k) {
    if (k < ppt && ((validmask >> k) & 1u)) {
      if (goes_new_audit<SPLIT>(pp, &S.ext, to_point(p[k]), near)) {
        acc_add(acc, p[k], FINAL);
        newmask |= 1u << k;
      }
    }
  }
  if (near) {  // some point passed the audit's integer filter: settle it with the real test (cold)
    near = false;
#pragma unroll
    for (int k = 0; k < kNarrowPPT; ++k)
      if (k < ppt && ((validmask >> k) & 1u)) near = near || recheck_near<SPLIT>(pp, &S.ext, to_point(p[k]));
  }
  uint64_t v[kAccWords];
  acc_words(acc, v);
  v[kAccPts] += (uint64_t)near << 32;  // tie audit (split_near_warp0)
  constexpr int WORDS = FINAL ? kAccWords : 5;
  reduce_stage1<WORDS>(S, v, nwarps, t, sync);
  if (t < 32) {
    reduce_stage2_warp0<WORDS>(S, nwarps);
    split_near_warp0(S, t);
    if (t == 0 && S.near) S.job_tie |= SPLIT ? (uint32_t)kTieCut : (uint32_t)kTieHyperplane;
    if (!FINAL) {
      // Fixed point of the local 2-means: the next pass's parameters are a function of {cnt, R, G, B} only, so
      // equal sums in two consecutive passes mean every later pass repeats this one exactly -- the remaining
      // iterations can be skipped without changing a bit of the result (the caller goes straight to the last pass).
      if (t == 0) {
        bool same = !SPLIT;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          same = same && (S.prev_tot[w] == S.tot[w]);
          S.prev_tot[w] = S.tot[w];
        }
        S.converged = same ? 1 : 0;
      }
      derive_params_warp0(S, jc, norm, t);
    }
  } else if (!FINAL) {
    derive_audit_warp1(S, jc, &S.aud, norm, nwarps, t);
  }
  sync();
  return newmask;
}

// This CTA's share of a wide job in one pass, seg[0 .. n_my): partial sums into v[].  Thread tid takes points
// tid + k * nthr, the same ones in every pass.  The first n_cached points live in cache[] for the rest of the round: the
// cut pass (SPLIT) loads every point from L2 and stores those, later passes read them back -- each thread only what it
// stored itself, so no barrier is needed -- and only the remainder comes from L2 again, four loads in flight per trip.
template <bool SPLIT, bool FINAL>
__device__ __forceinline__ void wide_classify(const PassParams &pp, const tie::PassExt *ext, uint32_t n_my, uint32_t nthr,
                                              const uint2 *seg, uint2 *cache, uint32_t n_cached, uint64_t (&v)[kAccWords]) {
  AccD acc = acc_zero();
  bool near = false;
  const uint32_t tid = threadIdx.x;
  if (tid < nthr) {
    uint32_t q = tid;
    if (!SPLIT) {
#pragma unroll 4
      for (; q < n_cached; q += nthr) {
        const uint2 p = cache[q];
        if (goes_new_audit<SPLIT>(pp, ext, to_point(p), near)) acc_add(acc, p, FINAL);
      }
    }
    for (; q < n_my; q += 4u * nthr) {
      uint2 raw[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t qq = q + (uint32_t)u * nthr;
        raw[u] = (qq < n_my) ? ld_cg_u2(seg + qq) : make_uint2(0u, 0u);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t qq = q + (uint32_t)u * nthr;
        if (SPLIT && qq < n_cached) cache[qq] = raw[u];
        if (qq < n_my && goes_new_audit<SPLIT>(pp, ext, to_point(raw[u]), near)) acc_add(acc, raw[u], FINAL);
      }
    }
  }
  if (near) {  // some point passed the audit's integer filter: settle it with the real test (cold; L2 holds the same bytes)
    near = false;
    for (uint32_t q = tid; q < n_my; q += nthr) near = near || recheck_near<SPLIT>(pp, ext, to_point(ld_cg_u2(seg + q)));
  }
  acc_words(acc, v);
  v[kAccPts] += (uint64_t)near << 32;  // tie audit (split_near_warp0)
}

// One narrow job, start to finish, on GT threads (the CTA, or one group): load its points into registers, run its passes
// to the fixed point, partition, write the children.  St = the job's state (Shared2 or a NarrowGroup), t = this thread's
// index among the GT, sync = their barrier.
template <int GT, typename St, typename Sync>
__device__ __forceinline__ void narrow_job(const SplitArgs &A, const Shared2 &S, St &G, const Arrays &R, int j, int child_base,
                                           int P, int t, Sync sync) {
  const int lane = t & 31;
  const int node = R.jobnode[j];
  if (t == 0) {
    const bool audit = A.tie_audit != 0u;
    G.cur = load_node(A, S, node);
    G.cur_old = 0;
    G.cur_new = 0;
    G.aud = job_audit_of(G.cur, audit);
    G.job_tie = (audit && tie::axis_tie(G.cur.tv, G.cur.eV)) ? (uint32_t)kTieAxis : 0u;  // D1 (:388-403)
  }
  sync();
  const JobConst jc = job_const_of(S, G.cur);
  // all warps the job has points for; up to kNarrowPPT points per thread, held in registers for every pass
  const uint32_t nthr = min((uint32_t)GT, max(32u, (jc.size + 31u) & ~31u));
  const int nwarps = (int)(nthr >> 5);
  uint2 p[kNarrowPPT];
  unsigned validmask = 0;
#pragma unroll
  for (int k = 0; k < kNarrowPPT; ++k) {
    const uint32_t off = (uint32_t)k * nthr + (uint32_t)t;
    p[k] = make_uint2(0, 0);
    if ((uint32_t)t < nthr && off < jc.size) {
      p[k] = ld_cg_u2(A.pts[jc.buf] + jc.begin + off);
      validmask |= 1u << k;
    }
  }
  set_split_params(S, G, jc, &G.aud, t);
  sync();
  const int ppt = (int)((jc.size + nthr - 1) / nthr);
  unsigned newmask = narrow_pass<true, false>(G, p, validmask, ppt, nwarps, jc, A.norm, t, sync);
  int pass = 1;
  for (; pass < P; ++pass) {
    newmask = narrow_pass<false, false>(G, p, validmask, ppt, nwarps, jc, A.norm, t, sync);
    if (G.converged) {  // uniform in the group: written before the barrier that ends the pass
      ++pass;
      break;
    }
  }
  newmask = narrow_pass<false, true>(G, p, validmask, ppt, nwarps, jc, A.norm, t, sync);
  trace2(A, kTraceNarrowJob, pass + 1);  // passes run, the cut pass and the final one included
  // G.tot = totals of the last pass; newmask = membership decided by it
  const uint32_t size_old = jc.size - (uint32_t)G.tot[kAccPts];
  if ((uint32_t)t < nthr) {
#pragma unroll
    for (int k = 0; k < kNarrowPPT; ++k) {
      const bool valid = (validmask >> k) & 1u;
      const bool to_new = (newmask >> k) & 1u;
      const unsigned m_new = __ballot_sync(0xffffffffu, to_new);
      const unsigned m_old = __ballot_sync(0xffffffffu, valid && !to_new);
      uint32_t base_new = 0, base_old = 0;
      if (lane == 0) {
        if (m_new) base_new = atomicAdd(&G.cur_new, (uint32_t)__popc(m_new));
        if (m_old) base_old = atomicAdd(&G.cur_old, (uint32_t)__popc(m_old));
      }
      base_new = __shfl_sync(0xffffffffu, base_new, 0);
      base_old = __shfl_sync(0xffffffffu, base_old, 0);
      if (valid) {
        const unsigned below = (1u << lane) - 1u;
        const uint32_t dst = to_new ? jc.begin + size_old + base_new + __popc(m_new & below)
                                    : jc.begin + base_old + __popc(m_old & below);
        A.pts[jc.buf ^ 1][dst] = p[k];
      }
    }
  }
  write_children(A, G, node, child_base + 2 * j, jc, G.job_tie, t);
  sync();
}

// Dynamic shared memory of the integer path (Shared2 + the arrays of Arrays), 16-B aligned.  The wide-point cache
// (Split2Extra::wide_cache_points) starts at this offset and takes whatever the launch reserves beyond it.
__host__ __device__ size_t split2_smem_bytes(uint32_t K, uint32_t cap) {
  size_t s = (sizeof(Shared2) + 15) & ~size_t(15);
  s += (size_t)cap * (8 + 4 + 4 + 4 + 4);
  s += (size_t)K * (8 + 4 + 4 + 4);
  s += (size_t)(K + 1) * 4 * 3;
  s += (size_t)K * 2 * 2;
  s += (size_t)K + 16 + (size_t)cap * (8 + 4);  // tie audit: jobtie, terr, byrank
  return (s + 64 + 15) & ~size_t(15);
}

// ---------------------------------------------------------------------------------------------------------
// The kernel
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(T, 65536 / (128 * T)) split2_kernel(const SplitArgs A, const Split2Extra X) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Shared2 &S = *reinterpret_cast<Shared2 *>(smem_raw);
  const int K = (int)A.num_colors, P = A.max_iters, G = (int)gridDim.x, b = (int)blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31;
  const uint32_t cap = A.node_cap;

  Arrays R;
  {
    unsigned char *cur = smem_raw + ((sizeof(Shared2) + 15) & ~size_t(15));
    R.tse = reinterpret_cast<double *>(cur);
    cur += (size_t)cap * 8;
    R.ctse = reinterpret_cast<double *>(cur);
    cur += (size_t)K * 8;
    R.child = reinterpret_cast<int32_t *>(cur);
    cur += (size_t)cap * 4;
    R.size = reinterpret_cast<uint32_t *>(cur);
    cur += (size_t)cap * 4;
    R.parent = reinterpret_cast<int32_t *>(cur);
    cur += (size_t)cap * 4;
    R.rank = reinterpret_cast<int32_t *>(cur);
    R.wprev = reinterpret_cast<uint64_t(*)[4]>(cur);
    cur += (size_t)cap * 4;
    R.jobnode = reinterpret_cast<int32_t *>(cur);
    cur += (size_t)K * 4;
    R.cnode = reinterpret_cast<int32_t *>(cur);
    cur += (size_t)K * 4;
    R.cand = reinterpret_cast<int32_t *>(cur);
    R.wfin = R.cand;
    cur += (size_t)K * 4;
    R.tile0 = reinterpret_cast<uint32_t *>(cur);
    cur += (size_t)(K + 1) * 4;
    R.slot0 = reinterpret_cast<uint32_t *>(cur);
    cur += (size_t)(K + 1) * 4;
    R.nidx = reinterpret_cast<uint32_t *>(cur);
    cur += (size_t)(K + 1) * 4;
    R.mywide = reinterpret_cast<uint16_t *>(cur);
    cur += (size_t)K * 2;
    R.mynarrow = reinterpret_cast<uint16_t *>(cur);
    cur += (size_t)K * 2;
    R.jobtie = reinterpret_cast<uint8_t *>(cur);
    cur += (size_t)K;
    cur = smem_raw + (((size_t)(cur - smem_raw) + 15) & ~size_t(15));
    R.terr = reinterpret_cast<double *>(cur);
    cur += (size_t)cap * 8;
    R.byrank = reinterpret_cast<int32_t *>(cur);
    R.wcache = reinterpret_cast<uint2 *>(smem_raw + split2_smem_bytes((uint32_t)K, cap));
  }
  const bool audit = A.tie_audit != 0u;

  const uint32_t U = A.num_points_dev ? ld_cg_u32(A.num_points_dev) : A.num_points;
  unsigned int bar_target = 0;
  trace2(A, kTraceBegin, 0);
  if (A.exact_small_max != 0u && U <= A.exact_small_max) {
    // small input: the reference's own summation order (dq_split_exact.cuh); stand-alone kernels did it unless fused
    if (X.exact_fused && U > 0u) {
      __shared__ SplitArgs s_args;
      __shared__ Split2Extra s_extra;
      if (tid == 0) {
        s_args = A;
        s_extra = X;
      }
      __syncthreads();
      exact_first_seen(X.exact_src, X.exact_first_seen, (uint32_t)(b * T + tid), (uint32_t)(G * T));
      if (X.exact_fused == 2u && (U > (uint32_t)exact::kSmemPoints || (K >= 32 && U >= 32u))) {
        // (few splits of a small input -- few clusters or few colours: CTA 0 alone, with everything in shared memory, is
        // quicker)
        // all CTAs: controller on CTA 0, the others split leaves ahead of it (dq_split_ordered.cuh)
        const ordered::Scratch og = ordered::carve(X.exact_scratch, A.node_cap);
        for (uint32_t i = (uint32_t)(b * T + tid); i < A.node_cap; i += (uint32_t)(G * T)) og.state[i] = ordered::kInvalid;
        if (b == 0 && tid < 4) og.counters[tid] = 0u;
        grid_barrier2(A, bar_target, X.progress);
        // (the bodies of the ordered path are not inlined: they get the argument blocks through shared memory, so that the
        // kernel parameters never have to be spilled to a local copy that the exact-integer path would then read too)
        ordered::run(s_args, s_extra, (int)U, smem_raw, b, G, bar_target);
        if (b == 0) publish_mailbox(A, U);
        return;
      }
      grid_barrier2(A, bar_target, X.progress);
      if (b == 0) {
        const size_t Kz = (size_t)K;
        exact::split_exact_body<T>(s_args, (int)U, smem_raw, X.exact_scratch, X.collect_uniq, X.collect_table, X.exact_first_seen, X.exact_f64,
                                   X.exact_f64 + Kz, X.exact_f64 + 2 * Kz, X.exact_f64 + 5 * Kz, X.exact_i32);
        publish_mailbox(A, U);
      }
    }
    return;
  }

  // ---- global statistics of all points (DivQuantClusterInitMeanAndVar, :60-104) + scratch reset ----
  {
    uint64_t v[kAccWords] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (X.collect_uniq != nullptr) {
      // four colours per thread and trip, a grid stride apart: all loads of a trip are issued before the first store
      // (the colours are distinct, which the compiler cannot know), so a trip costs one dependent pair of round trips
      constexpr int kCollect = 4;
      const size_t stride = (size_t)G * T;
      for (size_t base = (size_t)b * T + tid; base < U; base += kCollect * stride) {
        uint32_t c[kCollect], cnt[kCollect];
#pragma unroll
        for (int q = 0; q < kCollect; ++q) c[q] = (base + q * stride < U) ? __ldcs(X.collect_uniq + base + q * stride) : 0u;
#pragma unroll
        for (int q = 0; q < kCollect; ++q) cnt[q] = (base + q * stride < U) ? __ldcg(X.collect_table + c[q]) : 0u;
#pragma unroll
        for (int q = 0; q < kCollect; ++q) {
          if (base + q * stride < U) {
            X.collect_table[c[q]] = 0u;  // the count table is all-zero again when the kernel ends
            const uint2 p = make_uint2(c[q], cnt[q]);
            A.pts[0][base + q * stride] = p;
            add_point(v, p, true);
          }
        }
      }
    } else {
      for (size_t i = (size_t)b * T + tid; i < U; i += (size_t)G * T) add_point(v, ld_cg_u2(A.pts[0] + i), true);
    }
    trace2(A, kTraceCollected, 0);
    block_total<kAccWords>(S, v);
    if (tid < kAccWords && S.tot[tid] != 0)
      atomicAdd(reinterpret_cast<unsigned long long *>(A.root_acc + tid), (unsigned long long)S.tot[tid]);
    const size_t slot_words = (size_t)2 * X.slot_cap * kAccWords;
    for (size_t i = (size_t)b * T + tid; i < slot_words; i += (size_t)G * T) X.slots[i] = 0ull;
  }
  trace2(A, kTraceReduced, 0);
  grid_barrier2(A, bar_target);
  trace2(A, kTraceRootBarrier, 0);
  trace2(A, kTraceRoot, 0);

  if (A.cut_overrides != nullptr && (uint32_t)tid < min(A.num_cut_overrides, kCutOverrideCap)) S.ovr[tid] = A.cut_overrides[tid];
  if (tid == 0) {
    SplitNode root;
    root.tw = 1.0;  // weight[0] = 1.0 (:343)
    for (int c = 0; c < 3; ++c) {
      root.tm[c] = fmul(__ull2double_rn(ld_cg_u64(A.root_acc + kAccR + c)), A.norm);  // (:107-112)
      root.tv[c] = fsub(fmul(__ull2double_rn(ld_cg_u64(A.root_acc + kAccRR + c)), A.norm), fsq(root.tm[c]));
    }
    root.tse = 0.0;
    root.cut = 0.0;
    root.begin = 0;
    root.size = U;
    root.buf = 0;
    root.child = -1;
    root.axis = 0;
    root.parent = -1;
    root.eW = root.eS = root.eQ = root.eM = root.eV = root.eT = 0.0;
    root.tie = root.pad = 0u;
    if (audit) {
      const tie::Bounds rb = tie::root_bounds((double)U, root.tm, root.tv);
      root.eW = rb.eW, root.eS = rb.eS, root.eQ = rb.eQ, root.eM = rb.eM, root.eV = rb.eV, root.eT = rb.eT;
    }
    S.root = root;
    if (b == 0) A.nodes[0] = root;
    S.tie_total = 0u;
    S.cut_count = 0u;
    S.n_ovr = (A.cut_overrides != nullptr) ? min(A.num_cut_overrides, kCutOverrideCap) : 0u;
    R.terr[0] = 0.0;
    R.tse[0] = __longlong_as_double(0x7ff0000000000000ll);  // +inf: the first split is unconditional
    R.child[0] = -1;
    R.size[0] = U;
    R.parent[0] = -1;
    S.num_points = U;
    S.n_nodes = 1;
    S.n_prev = 1;  // nothing to absorb in round 0: the root's entries above are final (its TSE key is +inf)
    S.njobs = 0;
    S.prev_njobs = 0;
    S.mode = 0;
    S.done = 0;
    S.new_index = 1;
    S.old_index = 0;
  }
  __syncthreads();

  for (int round = 0;; ++round) {
    if (cta_error(A, S)) break;  // somebody's wait expired
    trace2(A, kTraceRoundBegin, round);
    // ================= controller (replicated) =================
    // (a) absorb the children created in the previous round
    {
      const int n_prev = S.n_prev, n_now = S.n_nodes;
      for (int i = n_prev + tid; i < n_now; i += T) {
        const SplitNode *nd = A.nodes + i;
        R.tse[i] = __ldcg(&nd->tse);
        R.terr[i] = __ldcg(&nd->eT);
        R.size[i] = __ldcg(&nd->size);
        R.child[i] = -1;
        R.parent[i] = R.jobnode[(i - n_prev) >> 1];
      }
      for (int j = tid; j < S.prev_njobs; j += T) R.child[R.jobnode[j]] = n_prev + 2 * j;
    }
    __syncthreads();
    trace2(A, kTracePhaseA, S.prev_njobs);

    // (b) which leaves to split next
    if (K <= 1) {
      if (tid == 0) S.done = 1;
      __syncthreads();
    } else if (S.mode == 0) {
      const int n_now = S.n_nodes, lo = (round == 0) ? 0 : S.n_prev;
      const bool need_count = n_now > K - 1;
      if (tid == 0) S.njobs = 0;
      __syncthreads();
      ordered_compact(
          S, lo, n_now,
          [&](int i) {
            const double t = R.tse[i];
            if (!(t > DBL_MIN)) return false;
            if (!need_count) return true;
            int above = 0;
            for (int m2 = 0; m2 < n_now; ++m2) above += (R.tse[m2] > t);
            return above < K - 1;
          },
          [&](int pos, int i) {
            if (pos < K) R.jobnode[pos] = i;
          },
          &S.njobs);
      __syncthreads();
      // node slots: the threshold policy may use the lower half, the sequential policy needs the rest
      // (many equal TSEs could also request more than K leaves at once: let the exact scan decide then)
      if (S.njobs > K || (S.njobs > 0 && (uint32_t)(S.n_nodes + 2 * S.njobs) > cap / 2)) {
        if (tid == 0) {
          if (audit) S.tie_total |= (uint32_t)kTieReplay;
          S.mode = 1;
          R.cnode[0] = 0;
          R.ctse[0] = 0.0;
        }
        __syncthreads();
      } else if (S.njobs == 0) {
        fast_assignment(A, S, R);
        if (S.bad) {
          if (tid == 0) {
            if (audit) S.tie_total |= (uint32_t)kTieReplay;
            S.mode = 1;
            R.cnode[0] = 0;
            R.ctse[0] = 0.0;
          }
        } else if (tid == 0) {
          S.done = 1;
        }
        __syncthreads();
      }
    }
    if (K > 1 && S.mode == 1 && !S.done) sequential_controller(A, S, R);
    trace2(A, kTracePhaseB, S.njobs);

    if (S.done) {
      if (b == 0) {
        emit_palette(A, S, R);
        if (tid == 0) {
          A.ctl[kCtlTie] = S.tie_total;
          A.ctl[kCtlDone] = 1;
          A.ctl[kCtlNodes] = (uint32_t)S.n_nodes;
          A.ctl[kCtlRounds] = (uint32_t)round;
        }
        publish_mailbox(A, U);
      }
      break;
    }
    if ((uint32_t)(S.n_nodes + 2 * S.njobs) > cap || (unsigned)(1 + (round + 1) * (P + 1)) > 0xFFFFu) {
      if (b == 0 && tid == 0) A.ctl[kCtlError] = 1;
      break;
    }

    // (c) work decomposition of this round
    const int njobs = S.njobs;
    for (int j = tid; j < njobs; j += T) {
      const uint32_t sz = R.size[R.jobnode[j]];
      const bool wide = sz > kNarrowMax;
      const uint32_t tiles = wide ? (sz + kWideTile - 1) / kWideTile : 0u;
      R.tile0[j] = tiles;
      R.nidx[j] = wide ? 0u : 1u;
      R.jobtie[j] = 0;
    }
    __syncthreads();
    block_scan(S, R.tile0, njobs);
    if (tid == 0) {
      R.tile0[njobs] = (uint32_t)S.scan_carry;
      S.nwide_tiles = S.scan_carry;
    }
    __syncthreads();
    // Wide tiles are dealt to the CTAs in contiguous blocks of the round's tile sequence (sizes differ by at most one),
    // so a job spans as few CTAs as possible: with few CTAs per frame (frame pipeline) a CTA then takes part in two
    // or three jobs per pass instead of all of them, and a CTA's share of a job is one contiguous range of points.
    const uint32_t tq = (uint32_t)S.nwide_tiles / (uint32_t)G, tr = (uint32_t)S.nwide_tiles % (uint32_t)G;
    auto cta_start = [&](uint32_t c) -> uint32_t { return c * tq + min(c, tr); };  // first tile of CTA c
    auto tile_owner = [&](uint32_t g) -> uint32_t {
      return (g < tr * (tq + 1u)) ? g / (tq + 1u) : tr + (g - tr * (tq + 1u)) / max(tq, 1u);
    };
    for (int j = tid; j < njobs; j += T) {
      const uint32_t g0 = R.tile0[j], g1 = R.tile0[j + 1];
      R.slot0[j] = (g1 > g0) ? tile_owner(g1 - 1u) - tile_owner(g0) + 1u : 0u;  // participants of the job
    }
    __syncthreads();
    block_scan(S, R.slot0, njobs);
    if (tid == 0) R.slot0[njobs] = (uint32_t)S.scan_carry;
    block_scan(S, R.nidx, njobs);
    if (tid == 0) {
      R.nidx[njobs] = (uint32_t)S.scan_carry;
      S.n_mywide = 0;
      S.n_mynarrow = 0;
    }
    __syncthreads();
    if (R.slot0[njobs] > X.slot_cap) {
      if (b == 0 && tid == 0) A.ctl[kCtlError] = 2;
      break;
    }
    const int child_base = S.n_nodes;
    const int nwide_tiles = S.nwide_tiles;
    ordered_compact(
        S, 0, njobs,
        [&](int j) {
          const uint32_t g0 = R.tile0[j], g1 = R.tile0[j + 1];
          if (g1 == g0) return false;
          return tile_owner(g0) <= (uint32_t)b && (uint32_t)b <= tile_owner(g1 - 1u);
        },
        [&](int pos, int j) { R.mywide[pos] = (uint16_t)j; }, &S.n_mywide);
    ordered_compact(
        S, 0, njobs,
        [&](int j) {
          if (R.nidx[j + 1] == R.nidx[j]) return false;
          return (int)(((uint32_t)nwide_tiles + R.nidx[j]) % (uint32_t)G) == b;
        },
        [&](int pos, int j) { R.mynarrow[pos] = (uint16_t)j; }, &S.n_mynarrow);
    __syncthreads();
    if (tid == 0) {
      S.prev_njobs = njobs;
      S.n_prev = S.n_nodes;
      S.n_nodes += 2 * njobs;
      if (b == 0) {
        A.ctl[kCtlSplits] += (uint32_t)njobs;
        A.ctl[kCtlJobs] = (uint32_t)njobs;
      }
    }
    const int n_mywide = S.n_mywide, n_mynarrow = S.n_mynarrow;
    for (int mw = tid; mw < n_mywide; mw += T) R.wfin[mw] = 0;
    for (int mw = tid; mw < min(n_mywide, kAudCache); mw += T) {
      // (executed by a few threads) constants of the first few wide jobs stay in shared memory
      const SplitNode nd = load_node(A, S, R.jobnode[R.mywide[mw]]);
      if (mw < kWideCache) S.wide[mw] = job_const_of(S, nd);
      S.wide_aud[mw] = job_audit_of(nd, audit);
      if (audit && tie::axis_tie(nd.tv, nd.eV)) R.jobtie[R.mywide[mw]] |= (uint8_t)kTieAxis;  // D1 (:388-403)
    }
    __syncthreads();
    trace2(A, kTracePhaseC, njobs);
    DQ_PROGRESS(round * 10000 + 1000 + n_mywide * 10 + n_mynarrow);

    // ================= wide jobs: all passes, partial sums exchanged through tagged slots =================
    // A CTA's share of a wide job = a contiguous run of its kWideTile-point tiles, classified by the warps it has
    // points for (wide_classify).
    const unsigned seq0 = 1u + (unsigned)round * (unsigned)(P + 1);
    auto wide_const = [&](int mw) -> JobConst {
      if (mw < kWideCache) return S.wide[mw];
      return job_const_of(S, load_node(A, S, R.jobnode[R.mywide[mw]]));
    };
    // This CTA's share of wide job j: participants, my rank among them, my first point and how many.
    struct Share {
      uint32_t m, me, first_point, n_my;
    };
    auto share_of = [&](int j, uint32_t size) -> Share {
      const uint32_t g0 = R.tile0[j], g1 = R.tile0[j + 1];
      const uint32_t first = tile_owner(g0), last = tile_owner(g1 - 1u);
      Share sh;
      sh.m = last - first + 1u;
      sh.me = (uint32_t)b - first;
      const uint32_t lo = max(g0, cta_start((uint32_t)b)) - g0, hi = min(g1, cta_start((uint32_t)b + 1u)) - g0;  // my tiles of it
      sh.first_point = lo * kWideTile;
      sh.n_my = min(hi * kWideTile, size) - sh.first_point;
      return sh;
    };
    // The points of a CTA's shares do not change during a round: the cut pass puts them into R.wcache, back to back
    // in mywide order (job mw from `base` on), and the later passes and the partition read the first n_cached of each share
    // from there.  Only what does not fit (few CTAs per frame, large K) is read from L2 in every pass.
    auto n_cached_of = [&](uint32_t base, uint32_t n_my) { return X.wide_cache_points > base ? min(n_my, X.wide_cache_points - base) : 0u; };
    // Fixed-point exit: every participant gathers the same totals, so each of them finds on its own
    // that {cnt, R, G, B} repeat the previous pass's -- the next parameters, and so every later classification, repeat
    // that pass exactly -- and runs this pass as the final one, as a narrow job does.  The participants therefore all
    // publish their final sums in the same pass and nobody writes the job's slots afterwards: the two slot buffers stay
    // enough, the final sums simply sit in the buffer and under the tag of that pass (R.wfin).
    int n_running = n_mywide;  // CTA-uniform
    for (int pass = 0; pass <= P && n_running > 0; ++pass) {
      unsigned long long *slots_w = X.slots + (size_t)(pass & 1) * X.slot_cap * kAccWords;
      const unsigned long long *slots_r = X.slots + (size_t)((pass & 1) ^ 1) * X.slot_cap * kAccWords;
      uint32_t base = 0;
      for (int mw = 0; mw < n_mywide; ++mw) {
        const int j = R.mywide[mw];
        const Share sh = share_of(j, R.size[R.jobnode[j]]);
        const uint32_t n_cached = n_cached_of(base, sh.n_my);
        uint2 *const cache = R.wcache + base;
        base += sh.n_my;
        if (R.wfin[mw] != 0) continue;
        const JobConst jc = wide_const(mw);
        const int m = (int)sh.m;
        const uint32_t me = sh.me;
        const uint32_t n_my = sh.n_my;
        const uint32_t nthr = min((uint32_t)T, (n_my + 31u) & ~31u);  // spread over as many warps as there are points for
#ifdef DQ_PROFILE_NARROW
        const long long w0 = clock64();
        long long w1 = w0;
#endif
        const JobAudit *aud = (mw < kAudCache) ? &S.wide_aud[mw] : nullptr;
        if (pass == 0) {
          set_split_params(S, S, jc, aud);
        } else {
          gather(A, S, slots_r, R.slot0[j], m, 5, (seq0 + pass - 1) & 0xFFFFu);
          if (tid == 0 && S.near) R.jobtie[j] |= (pass == 1) ? (uint8_t)kTieCut : (uint8_t)kTieHyperplane;
#ifdef DQ_PROFILE_NARROW
          w1 = clock64();
#endif
          derive_params_warp0(S, jc, A.norm);
          derive_audit_warp1(S, jc, aud, A.norm, kWarps);
          if (tid == 0 && pass < P) {
            bool same = pass >= 2;  // (pass 1 gathers the cut pass's sums)
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              same = same && (R.wprev[mw][w] == S.tot[w]);
              R.wprev[mw][w] = S.tot[w];
            }
            S.converged = same ? 1 : 0;
          }
        }
        __syncthreads();
#ifdef DQ_PROFILE_NARROW
        const long long w2 = clock64();
#endif
        const bool fin = pass == P || (pass >= 2 && S.converged != 0);  // CTA-uniform
        const PassParams pp = S.pp;
        uint64_t v[kAccWords];
        {
          const uint2 *seg = A.pts[jc.buf] + jc.begin + sh.first_point;
          if (pass == 0) wide_classify<true, false>(pp, &S.ext, n_my, nthr, seg, cache, n_cached, v);
          else if (fin) wide_classify<false, true>(pp, &S.ext, n_my, nthr, seg, cache, n_cached, v);
          else wide_classify<false, false>(pp, &S.ext, n_my, nthr, seg, cache, n_cached, v);
        }
#ifdef DQ_PROFILE_NARROW
        const long long w3 = clock64();
#endif
        if (fin) {
          --n_running;
          if (tid == 0) R.wfin[mw] = pass + 1;
          if (tid == 0 && mw < kWideCache) S.wide_pp[mw] = pp;
          reduce_stage1<kAccWords>(S, v, (int)(nthr >> 5));
          if (tid < 32) {
            reduce_stage2_warp0<kAccWords>(S, (int)(nthr >> 5));
            publish<kAccWords>(slots_w, R.slot0[j] + me, S, (seq0 + pass) & 0xFFFFu);
          }
        } else {
          reduce_stage1<5>(S, v, (int)(nthr >> 5));
#ifdef DQ_PROFILE_NARROW
          if (tid == 0 && pass > 0) atomicAdd(X.progress + 769, (uint32_t)(clock64() - w3));  // stage 1 + sync
#endif
          if (tid < 32) {
#ifdef DQ_PROFILE_NARROW
            const long long w4 = clock64();
#endif
            reduce_stage2_warp0<5>(S, (int)(nthr >> 5));
#ifdef DQ_PROFILE_NARROW
            const long long w5 = clock64();
#endif
            publish<5>(slots_w, R.slot0[j] + me, S, (seq0 + pass) & 0xFFFFu);
#ifdef DQ_PROFILE_NARROW
            if (tid == 0 && pass > 0) {
              atomicAdd(X.progress + 770, (uint32_t)(w5 - w4));          // stage 2
              atomicAdd(X.progress + 771, (uint32_t)(clock64() - w5));   // publish
            }
#endif
          }
        }
#ifdef DQ_PROFILE_NARROW
        const long long w6 = clock64();
#endif
        __syncthreads();
#ifdef DQ_PROFILE_NARROW
        if (tid == 0 && pass > 0) atomicAdd(X.progress + 772, (uint32_t)(clock64() - w6));  // closing barrier
        if (tid == 0 && pass > 0) atomicAdd(X.progress + 768, (uint32_t)(w3 - w2));  // classification only
        if (tid == 0 && pass > 0) {
          atomicAdd(X.progress + 764, (uint32_t)(w1 - w0));            // gather (wait + reduce)
          atomicAdd(X.progress + 765, (uint32_t)(w2 - w1));            // derive + sync
          atomicAdd(X.progress + 766, (uint32_t)(clock64() - w2));     // classify + reduce + publish
          atomicAdd(X.progress + 767, 1u);
        }
#endif
      }
      if (n_mywide) trace2(A, kTracePass, pass);
      DQ_PROGRESS(round * 10000 + 2000 + pass);
    }
    // partition of the wide jobs + children
    uint32_t base = 0;
    for (int mw = 0; mw < n_mywide; ++mw) {
      const int j = R.mywide[mw];
      const JobConst jc = wide_const(mw);
      const Share sh = share_of(j, jc.size);
      const uint32_t n_cached = n_cached_of(base, sh.n_my);
      const uint2 *const cache = R.wcache + base;
      base += sh.n_my;
      const int m = (int)sh.m;
      const uint32_t me = sh.me;
      const int pf = R.wfin[mw] - 1;  // the job's final pass
      // classification of the final pass (parameters from the totals of pass pf-1)
      if (mw >= kWideCache) {
        gather(A, S, X.slots + (size_t)((pf - 1) & 1) * X.slot_cap * kAccWords, R.slot0[j], m, 5, (seq0 + pf - 1) & 0xFFFFu);
        derive_params_warp0(S, jc, A.norm);  // (only the partition's re-classification follows: no audit)
        __syncthreads();
      }
      const PassParams pp = (mw < kWideCache) ? S.wide_pp[mw] : S.pp;
      __syncthreads();
      const unsigned long long *slots_p = X.slots + (size_t)(pf & 1) * X.slot_cap * kAccWords;
      gather(A, S, slots_p, R.slot0[j], m, kAccWords, (seq0 + pf) & 0xFFFFu);
      if (tid == 0 && S.near) R.jobtie[j] |= (uint8_t)kTieHyperplane;
      __syncthreads();
      if (S.tot[kAccPts] > jc.size) continue;  // only after an expired wait: never scatter out of the segment
      const uint32_t size_old = jc.size - (uint32_t)S.tot[kAccPts];
      // Destinations without atomics: the participants' new-side counts of the last pass are in the slots just
      // gathered, so the CTAs ranked before this one fix where its points start in both halves
      // (deterministic, CTA-major order); inside the CTA a per-piece prefix over the warps does the rest.
      {
        // (shares are contiguous and in CTA order: the points before mine are simply those of the tiles before mine)
        uint32_t before_new = 0;
        for (uint32_t i = (uint32_t)tid; i < me; i += T)
          before_new += (uint32_t)(ld_relaxed_u64(slots_p + (size_t)(R.slot0[j] + i) * kAccWords + kAccPts) & kValueMask);
        before_new = __reduce_add_sync(0xffffffffu, before_new);
        if (lane == 0) S.part_new[tid >> 5] = before_new;
        __syncthreads();
        if (tid == 0) {
          uint32_t bn = 0;
          for (int w = 0; w < kWarps; ++w) bn += S.part_new[w];
          S.base_new = bn;
          S.base_old = sh.first_point - bn;
        }
        __syncthreads();
      }
      uint32_t run_new = S.base_new, run_old = S.base_old;
      int flip = 0;
      // (the cache was written by other threads in the cut pass: the barriers since then order it)
      const uint2 *seg = A.pts[jc.buf] + jc.begin + sh.first_point;
      auto point = [&](uint32_t q) { return q < n_cached ? cache[q] : ld_cg_u2(seg + q); };
      uint2 p_next = make_uint2(0, 0);
      if ((uint32_t)tid < sh.n_my) p_next = point(tid);
      for (uint32_t piece = 0; piece < sh.n_my; piece += T) {
        // T-point pieces of this CTA's (contiguous) share, in order; the next piece's points are already on their way
        const bool valid = piece + tid < sh.n_my;
        const uint2 p = p_next;
        if (piece + T + tid < sh.n_my) p_next = point(piece + T + tid);
        const bool to_new = valid && goes_new(pp, false, p.x);
        const unsigned m_new = __ballot_sync(0xffffffffu, to_new);
        const unsigned m_old = __ballot_sync(0xffffffffu, valid && !to_new);
        uint32_t *wn = S.piece_new[flip], *wo = S.piece_old[flip];  // double-buffered: one barrier per piece
        if (lane == 0) {
          wn[tid >> 5] = (uint32_t)__popc(m_new);
          wo[tid >> 5] = (uint32_t)__popc(m_old);
        }
        __syncthreads();
        uint32_t base_new = run_new, base_old = run_old, tot_new = 0, tot_old = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
          const uint32_t cn = wn[w], co = wo[w];
          if (w < (tid >> 5)) base_new += cn, base_old += co;
          tot_new += cn, tot_old += co;
        }
        run_new += tot_new;
        run_old += tot_old;
        flip ^= 1;
        if (valid) {
          const unsigned below = (1u << lane) - 1u;
          const uint32_t dst = to_new ? jc.begin + size_old + base_new + __popc(m_new & below)
                                      : jc.begin + base_old + __popc(m_old & below);
          A.pts[jc.buf ^ 1][dst] = p;
        }
      }
      if (me == 0) {  // owner: the CTA holding the job's first tile
        if (tid == 0) S.cur = load_node(A, S, R.jobnode[j]);
        __syncthreads();
        write_children(A, S, R.jobnode[j], child_base + 2 * j, jc, R.jobtie[j]);
      }
      __syncthreads();
    }
    if (n_mywide) trace2(A, kTracePartition, n_mywide);
    DQ_PROGRESS(round * 10000 + 3000);

    // ================= narrow jobs: everything inside this CTA =================
    // Jobs of more than kGroupMax points take the whole CTA, one after the other; the others run kGroups at a time, one per
    // group of kGroupWarps warps, each group taking the CTA's next such job as soon as it is free.
    for (int mn = 0; mn < n_mynarrow; ++mn) {
      const int j = R.mynarrow[mn];
      if (R.size[R.jobnode[j]] > kGroupMax) narrow_job<T>(A, S, S, R, j, child_base, P, tid, CtaSync());
    }
    if (n_mynarrow) {
      if (tid == 0) S.narrow_next = 0;
      __syncthreads();
      const int t = tid % kGroupT;
      NarrowGroup &G = S.grp[tid / kGroupT];
      const GroupSync gsync{1 + tid / kGroupT};
      for (;;) {
        if (t == 0) {
          int k;
          do {
            k = atomicAdd(&S.narrow_next, 1);
          } while (k < n_mynarrow && R.size[R.jobnode[R.mynarrow[k]]] > kGroupMax);
          G.next = k;
        }
        gsync();
        const int k = G.next;  // (rewritten only after the job's closing barrier)
        if (k >= n_mynarrow) break;
        narrow_job<kGroupT>(A, S, G, R, R.mynarrow[k], child_base, P, t, gsync);
      }
      __syncthreads();
    }
    if (n_mynarrow) trace2(A, kTracePartition, 1000 + n_mynarrow);
    DQ_PROGRESS(round * 10000 + 4000);

    grid_barrier2(A, bar_target, X.progress);
    trace2(A, kTraceCtlBarrier, round);
  }
}

}  // namespace

size_t split2_slot_capacity(uint32_t point_capacity, uint32_t num_colors, int sm_count) {
  // every wide job needs min(tiles, CTAs) slots; wide tiles <= points / kWideTile + jobs
  (void)sm_count;
  return (size_t)point_capacity / kWideTile + num_colors + 64;
}

// CTAs of the split kernel that can be co-resident on the device (cooperative launch limit) for this K.
int split2_max_ctas(int sm_count, uint32_t num_colors) {
  // (occupancy and the raised shared-memory limit belong to the device: keyed by device ordinal as well)
  static std::mutex mu;
  static std::map<std::pair<int, size_t>, int> cache;
  const size_t smem = split2_smem_bytes(num_colors, 8 * num_colors + 16);
  int dev = 0;
  DQ_CUDA_CHECK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(std::make_pair(dev, smem));
  if (it == cache.end()) {
    int per_sm = 0;
    DQ_CUDA_CHECK(cudaFuncSetAttribute(split2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max(smem, (size_t)(216 * 1024))));
    DQ_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, split2_kernel, T, smem));
    it = cache.emplace(std::make_pair(dev, smem), std::max(per_sm, 1)).first;
  }
  return it->second * sm_count;
}

SplitLaunch split2_plan(int requested_ctas, int sm_count, uint32_t num_colors) {
  SplitLaunch plan;
  const int cap = split2_max_ctas(sm_count, num_colors);
  plan.grid = (requested_ctas >= 1 && requested_ctas <= cap) ? requested_ctas : cap;
  // The small-input body lives in the same dynamic shared memory, and the integer path keeps its wide-job points in what
  // that body needs beyond the integer path's own arrays (one CTA per SM either way: 128 registers x 512).  Every launch
  // reserves it, fused small-input body or not.  (Not more: crossing the 196 KB carve-out step costs the frame pipeline
  // 10-40 %, DESIGN 5.5.)
  plan.smem_bytes = std::max(split2_smem_bytes(num_colors, 8 * num_colors + 16), split_exact_smem_bytes());
  return plan;
}

void split2_launch(const SplitArgs &args_in, const Split2Extra &extra, const SplitLaunch &plan, cudaStream_t stream) {
  SplitArgs args = args_in;
  args.node_cap = 8 * args.num_colors + 16;
  (void)split2_max_ctas(1, args.num_colors);  // raises the kernel's dynamic shared memory limit once
  Split2Extra x = extra;
  const size_t arrays = split2_smem_bytes(args.num_colors, args.node_cap);
  x.wide_cache_points = plan.smem_bytes > arrays ? (uint32_t)((plan.smem_bytes - arrays) / sizeof(uint2)) : 0u;
  void *kargs[] = {(void *)&args, (void *)&x};
  DQ_CUDA_CHECK(cudaLaunchCooperativeKernel((const void *)split2_kernel, dim3(plan.grid), dim3(T), kargs, plan.smem_bytes, stream));
}

}  // namespace dq

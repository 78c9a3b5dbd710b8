// dq_split_exact.cuh -- the divisive phase for SMALL inputs, in the reference's own summation order.
//
// Reference: DivQuantCluster<UW=false,...>, DivQuant/DivQuantCluster.cpp:133-1097 (weighted path) and
// DivQuantClusterInitMeanAndVar, :49-123.
//
// Why this exists.  In the weighted path the reference accumulates  weight_i * channel_i  as doubles, one point
// after the other, in the order calc_color_table emitted the unique colours (hash bucket ascending, most
// recently first-seen colour first inside a bucket, MapColors.cpp:157-198).  The large-input kernels
// (dq_split2.cu) use exact integer sums instead, which differ from those doubles by ~1e-16 relative.  That
// never matters unless a decision sits exactly on a tie -- a mean on an integer, two equal variances or TSEs --
// which is what small or synthetic inputs (few colours, equal counts, tiny clusters) produce.  There the
// reference decides by its own rounding noise, so to return its palette bit for bit the noise has to be
// reproduced: up to SplitArgs::exact_small_max (<= kExactMaxPoints) unique colours this code walks the reference's
// loop with the same sequential double accumulations (one lane per accumulator chain, non-contracted IEEE
// operations in the reference's order).  Up to 4096 points everything lives in shared memory; above, the point
// arrays live in a global scratch (L2) and only the staged terms and the per-cluster arrays stay on chip.
//
// One CTA.  Launched for every weighted call; returns at once when U is larger (the split kernels return at
// once when it is not), so no host round trip is needed to choose.
//
// Structure of one pass over the cluster being split (cur[0..cur_n), ascending original order):
//   select   every thread classifies a contiguous piece, an exclusive scan gives each new-side point its rank
//   terms    w*c (and w, w*c*c) of the new-side points are written to shared memory in rank order
//   chains   lane l < 7 of warp 0 adds terms[l][0..n) one after the other -- the reference's sum, add for add
//   scalars  lanes 0..2 derive the centres per channel, lane 0 the hyperplane
// Clusters of up to 512 points are handled by warp 0 alone (no block barriers inside the 11 passes).
#pragma once

#include "dq_split_math.cuh"

#include <cfloat>

namespace dq {
namespace exact {

constexpr int kSmemPoints = 4096;  // inputs up to this size keep their point arrays in shared memory
constexpr int kIndexBits = 18;     // sort key = bucket << 49 | (0x7FFFFFFF - first seen) << 18 | arrival index
constexpr int kTile = 1024;        // new-side points whose terms are staged at a time
constexpr int kSolo = 512;         // clusters up to this size are split by warp 0 alone
constexpr int kPiece = 16;         // consecutive points a thread classifies per chunk (bits of its mask)
constexpr int kSmemColors = 896;   // (keeps sizeof(Shared) below the 196 KB shared-memory carve-out step)
constexpr int kMaxChunks = 64;     // kExactMaxPoints / (256 threads * kPiece)
static_assert(kExactMaxPoints <= (1u << kIndexBits), "index bits of the sort key");
static_assert(kSolo <= kPiece * 32 && kSolo <= kTile, "a solo pass is one chunk and one tile");
static_assert(kExactMaxPoints <= 256u * kPiece * kMaxChunks, "chunk count");

struct Shared {
  union {
    unsigned long long keys[kSmemPoints];  // only while the points are put in order
    double terms[7][kTile];
  };
  double w[kSmemPoints];
  uint32_t colour[kSmemPoints];
  uint16_t member[kSmemPoints];
  uint32_t cur[kSmemPoints];
  // per-cluster arrays of the reference (:296-324) when K fits, else the global scratch is used
  double k_weight[kSmemColors], k_tse[kSmemColors], k_mean[3 * kSmemColors], k_var[3 * kSmemColors];
  int32_t k_size[kSmemColors];
  double chain[8];
  int32_t warp_tmp[32];
  double red_val[32];
  int32_t red_idx[32];
  int32_t cur_n, old_index, new_size, emitted, steady;
  // scalars of the current split
  double tw, tm[3], tv[3], nw, ow, nm[3], om[3], nv[3];
  double lhs, rr[3], cut;
  int32_t axis;
};

// One CTA of the split kernel per SM holds this much dynamic shared memory; above the 196 KB carve-out step the SM falls
// back to the 228 KB configuration, which cost the frame pipeline 10-40 % (measured), so stay below it.
static_assert(sizeof(Shared) <= 196 * 1024 - 4096, "keep the fused ordered path under the 196 KB shared-memory carve-out");

// The per-point arrays: shared memory (U <= kSmemPoints) or the global scratch.
struct Points {
  unsigned long long *keys;
  double *w;         // weights[] of calc_color_table (:172,185)
  uint32_t *colour;
  uint16_t *member;  // K <= kExactMaxColors <= 65535
  uint32_t *cur;     // points of the cluster being split, ascending original order (:929-1019)
  bool cur_shared_across_ctas;  // index lists written by other CTAs: read them past the (incoherent) L1
  bool in_global;    // the point arrays live in the global scratch: Shared::w/colour/member/cur are free (chunk_sums_parallel)
};
__device__ __forceinline__ int load_cur(const Points &P, int j) {
  return P.cur_shared_across_ctas ? (int)__ldcg(P.cur + j) : (int)P.cur[j];
}
// global scratch, shared layout of both forms: keys 8 | w 8 | colour 4 | index list 4 | second index list 4 | member 2 (+2)
constexpr size_t kScratchBytes = (size_t)kExactMaxPoints * 32;

__device__ __forceinline__ double chan(uint32_t p, int c) { return byte_to_double((p >> (16 - 8 * c)) & 0xFFu); }
__device__ __forceinline__ double chan_sq(uint32_t p, int c) {
  const uint32_t v = (p >> (16 - 8 * c)) & 0xFFu;
  return u52_to_double((uint64_t)(v * v));  // the reference squares in int, then converts (:98-100, :741-743)
}

// Do two values act alike as inputs of a split?  Equal bits -- or both NaN: sign and payload of a NaN reach no comparison
// (all false), no non-NaN result and no conversion (NaN -> 0), and the empty clusters of a K > U tail do carry NaNs whose
// sign flips from one split to the next.
__device__ __forceinline__ bool same_input(double a, double b) {
  return __double_as_longlong(a) == __double_as_longlong(b) || (a != a && b != b);
}

template <bool SOLO>
__device__ __forceinline__ void group_sync() {
  if (SOLO) __syncwarp();
  else __syncthreads();
}

__device__ __forceinline__ void store_terms(Shared &S, int slot, double wt, uint32_t p, int nchains) {
  S.terms[0][slot] = fmul(wt, chan(p, 0));
  S.terms[1][slot] = fmul(wt, chan(p, 1));
  S.terms[2][slot] = fmul(wt, chan(p, 2));
  S.terms[3][slot] = wt;
  if (nchains > 4) {
    S.terms[4][slot] = fmul(wt, chan_sq(p, 0));
    S.terms[5][slot] = fmul(wt, chan_sq(p, 1));
    S.terms[6][slot] = fmul(wt, chan_sq(p, 2));
  }
}

// lane l < nchains of warp 0 continues chain l over the n staged terms, in order
__device__ __forceinline__ void add_terms(Shared &S, int n, int nchains, double &acc) {
  const int t = threadIdx.x;
  if (t < nchains) {
    const double *src = S.terms[t];
    int j = 0;
    for (; j + 8 <= n; j += 8) {
      const double a0 = src[j], a1 = src[j + 1], a2 = src[j + 2], a3 = src[j + 3];
      const double a4 = src[j + 4], a5 = src[j + 5], a6 = src[j + 6], a7 = src[j + 7];
      acc = fadd(acc, a0);
      acc = fadd(acc, a1);
      acc = fadd(acc, a2);
      acc = fadd(acc, a3);
      acc = fadd(acc, a4);
      acc = fadd(acc, a5);
      acc = fadd(acc, a6);
      acc = fadd(acc, a7);
    }
    for (; j < n; ++j) acc = fadd(acc, src[j]);
  }
}

// Exclusive rank of this thread's `mine` items among the group's and the group's total.
template <int THREADS, bool SOLO>
__device__ __forceinline__ void group_ranks(Shared &S, int mine, bool flag, int &first, int &total, bool &any_flag) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  first = incl - mine;
  if (SOLO) {
    total = __shfl_sync(0xffffffffu, incl, 31);
    any_flag = __any_sync(0xffffffffu, flag);
  } else {
    __syncthreads();  // the previous reader of warp_tmp is done
    if (lane == 31) S.warp_tmp[warp] = incl;
    any_flag = __syncthreads_or(flag) != 0;
    total = 0;
    for (int q = 0; q < THREADS / 32; ++q) {
      if (q < warp) first += S.warp_tmp[q];
      total += S.warp_tmp[q];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// The reference's sequential double sums, evaluated in parallel.
//
// s <- RN(s + t) over the new-side terms of one chunk, for each of the `nchains` accumulator chains, starting from the
// chain's accumulator and giving exactly the value the one-term-after-the-other loop of add_terms gives.  Why that is
// possible: while the accumulator stays inside one binade [2^e, 2^(e+1)) every addition rounds to a multiple of
// q = 2^(e-52), and s (a multiple of q) + t rounds to s + RN_q(t) unless t's remainder is exactly q/2 (round-half-even
// looks at s then).  So inside a binade the sum of a run of terms is s + sum RN_q(t_i): an order-free exact sum.
//   phase A  every thread adds its piece's terms (plain doubles) and a block scan of those gives the approximate
//            accumulator at every piece: the binade e each piece runs in, or "unsafe" when the piece may cross into the
//            next binade (judged with a 2^-20 margin) or starts from zero
//   phase B  every thread adds RN_q(t) of its terms (C = 2^e: RN(C + t) - C, the residual t - that tells an exact half);
//            the terms of unsafe pieces (crossings, exact halves: a few per chunk) are staged instead
//   walk     thread c < nchains carries chain c's exact accumulator through the pieces: warps whose 32 pieces are safe
//            in one binade in one step, safe pieces in one step each, staged terms one by one.  Every step is checked
//            on the exact accumulator (it is in binade e before and after): a failed check abandons the chunk,
//            and the caller falls back to the staged sequential loop.  The result is therefore the sequential sum
//            unconditionally; the predictions only decide how fast it is reached.
// Uses Shared::terms (piece table) and Shared::w (staged terms): only when the point arrays live in global memory.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kParSlots = 36;     // staged (unsafe) pieces per chain and chunk
constexpr int kParMinTerms = 768; // chunks with fewer new-side terms take the sequential loop
constexpr uint32_t kMetaEmpty = 0u, kMetaMixed = 0xFFFFFFFFu, kMetaUnsafe = 0x80000000u;

__device__ __forceinline__ int exp_of(double x) { return (__double2hiint(x) >> 20) & 0x7FF; }  // biased; 0 for 0.0
__device__ __forceinline__ double pow2_biased(int e) { return __hiloint2double(e << 20, 0); }

template <int THREADS>
struct ParScratch {
  double pieceD[7][THREADS];
  uint32_t meta[7][THREADS];  // 0 nothing to add | biased exponent (safe) | kMetaUnsafe | slot << 8 | terms
  double warpD[7][THREADS / 32];
  uint32_t warpmeta[7][THREADS / 32];  // kMetaEmpty | exponent (every piece safe, one binade) | kMetaMixed
  double scan[7][THREADS / 32];
  uint32_t slots[8];  // [c] staged pieces of chain c, [7] failure flag
};
static_assert(sizeof(ParScratch<512>) <= sizeof(double) * 7 * kTile, "piece table must fit into Shared::terms");
static_assert(7 * kParSlots * kPiece <= kSmemPoints, "staged terms must fit into Shared::w");

template <int THREADS>
__device__ __noinline__ bool chunk_sums_parallel(Shared &S, const Points &P, int lo, int hi, unsigned mask, int nchains, double &acc) {
  ParScratch<THREADS> &Q = *reinterpret_cast<ParScratch<THREADS> *>(&S.terms[0][0]);
  double *const staged = S.w;  // [7][kParSlots * kPiece]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < nchains) S.chain[tid] = acc;
  if (tid < 8) Q.slots[tid] = 0u;
  // ---- phase A: plain sums of my piece ----
  double p[7];
#pragma unroll
  for (int c = 0; c < 7; ++c) p[c] = 0.0;
  for (int j = lo; j < hi; ++j) {
    if (!((mask >> (j - lo)) & 1u)) continue;
    const int idx = load_cur(P, j);
    const double wt = P.w[idx];
    const uint32_t col = P.colour[idx];
#pragma unroll
    for (int c = 0; c < 3; ++c) p[c] = fadd(p[c], fmul(wt, chan(col, c)));
    p[3] = fadd(p[3], wt);
    if (nchains > 4) {
#pragma unroll
      for (int c = 0; c < 3; ++c) p[4 + c] = fadd(p[4 + c], fmul(wt, chan_sq(col, c)));
    }
  }
  // ---- exclusive block scan of p[] ----
  double before[7];
#pragma unroll
  for (int c = 0; c < 7; ++c) {
    before[c] = 0.0;
    if (c < nchains) {
      double incl = p[c];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      if (lane == 31) Q.scan[c][warp] = incl;
      before[c] = incl - p[c];
    }
  }
  __syncthreads();
  // ---- binade of every piece, RN_q sums (phase B) ----
  int e[7];
  unsigned unsafe = 0, staged_done = 0;
  double D[7];
#pragma unroll
  for (int c = 0; c < 7; ++c) {
    D[c] = 0.0;
    e[c] = 0;
    if (c < nchains) {
      double a = S.chain[c] + before[c];
      for (int w = 0; w < warp; ++w) a += Q.scan[c][w];
      const double b = a + p[c];
      if (p[c] > 0.0) {
        const int ea = exp_of(a * (1.0 - 9.5367431640625e-07)), eb = exp_of(b * (1.0 + 9.5367431640625e-07));
        e[c] = ea;
        if (!(a > 0.0) || ea != eb || ea == 0) unsafe |= 1u << c;
      }
    }
  }
  for (int round = 0; round < 2; ++round) {
    // round 0: RN_q sums of the safe chains, terms of the chains known to be unsafe are staged
    // round 1: only if an exact half turned up in round 0 -- those chains are staged now
    const unsigned to_stage = unsafe & ~staged_done;
    int slot[7];
#pragma unroll
    for (int c = 0; c < 7; ++c) {
      slot[c] = 0;
      if (c < nchains && ((to_stage >> c) & 1u)) slot[c] = (int)atomicAdd(&Q.slots[c], 1u);
    }
    if (round == 1 && to_stage == 0u) break;
    int k = 0;
    unsigned halves = 0;
    for (int j = lo; j < hi; ++j) {
      if (!((mask >> (j - lo)) & 1u)) continue;
      const int idx = load_cur(P, j);
      const double wt = P.w[idx];
      const uint32_t col = P.colour[idx];
#pragma unroll
      for (int c = 0; c < 7; ++c) {
        if (c >= nchains) continue;
        const bool mine_staged = (to_stage >> c) & 1u;
        const bool mine_sum = round == 0 && p[c] > 0.0 && !((unsafe >> c) & 1u);
        if (!mine_staged && !mine_sum) continue;
        const double t = (c == 3) ? wt : ((c < 3) ? fmul(wt, chan(col, c)) : fmul(wt, chan_sq(col, c - 4)));
        if (mine_staged) {
          if (slot[c] < kParSlots) staged[(c * kParSlots + slot[c]) * kPiece + k] = t;
        } else {
          const double C = pow2_biased(e[c]);
          const double y = fsub(fadd(C, t), C);  // RN_q(t), q = ulp of binade e
          const double r = fsub(t, y);           // exact
          if (fabs(r) == pow2_biased(e[c] - 53)) halves |= 1u << c;  // exactly q/2: the accumulator's parity decides
          D[c] = fadd(D[c], y);
        }
      }
      ++k;
    }
    staged_done |= to_stage;
#pragma unroll
    for (int c = 0; c < 7; ++c) {
      if (c < nchains && ((to_stage >> c) & 1u)) {
        if (slot[c] >= kParSlots) Q.slots[7] = 1u;  // no room: abandon the chunk
        Q.meta[c][tid] = kMetaUnsafe | ((uint32_t)slot[c] << 8) | (uint32_t)k;
      }
    }
    unsafe |= halves;
    if (halves == 0u) break;
  }
  // ---- piece table + warp aggregates ----
#pragma unroll
  for (int c = 0; c < 7; ++c) {
    if (c < nchains) {
      const bool is_unsafe = (unsafe >> c) & 1u, empty = !(p[c] > 0.0);
      if (!is_unsafe) {
        Q.pieceD[c][tid] = D[c];
        Q.meta[c][tid] = empty ? kMetaEmpty : (uint32_t)e[c];
      }
      const int e_max = __reduce_max_sync(0xffffffffu, (empty || is_unsafe) ? 0 : e[c]);
      const bool uniform = __all_sync(0xffffffffu, !is_unsafe && (empty || e[c] == e_max));
      double dw = (empty || is_unsafe) ? 0.0 : D[c];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) dw = fadd(dw, __shfl_xor_sync(0xffffffffu, dw, o));
      if (lane == 0) {
        Q.warpD[c][warp] = dw;
        Q.warpmeta[c][warp] = !uniform ? kMetaMixed : (e_max == 0 ? kMetaEmpty : (uint32_t)e_max);
      }
    }
  }
  __syncthreads();
  // ---- walk: thread c carries chain c ----
  double s = acc;
  if (tid < nchains && Q.slots[7] == 0u) {
    const int c = tid;
    bool fail = false;
    for (int w = 0; w < THREADS / 32 && !fail; ++w) {
      const uint32_t wm = Q.warpmeta[c][w];
      if (wm == kMetaEmpty) continue;
      if (wm != kMetaMixed && exp_of(s) == (int)wm) {
        const double s2 = fadd(s, Q.warpD[c][w]);  // exact while it stays in the binade
        if (exp_of(s2) == (int)wm) {
          s = s2;
          continue;
        }
      }
      for (int i = w * 32; i < w * 32 + 32; ++i) {
        const uint32_t m = Q.meta[c][i];
        if (m == kMetaEmpty) continue;
        if (m & kMetaUnsafe) {
          const double *src = staged + (c * kParSlots + (int)((m >> 8) & 0xFFu)) * kPiece;
          const int n = (int)(m & 0xFFu);
          for (int k = 0; k < n; ++k) s = fadd(s, src[k]);
        } else {
          const double s2 = fadd(s, Q.pieceD[c][i]);
          if (exp_of(s) != (int)m || exp_of(s2) != (int)m) {
            fail = true;
            break;
          }
          s = s2;
        }
      }
    }
    if (fail) Q.slots[7] = 1u;
  }
  __syncthreads();
  const bool ok = Q.slots[7] == 0u;
  __syncthreads();  // the table is free again
  if (ok && tid < nchains) acc = s;
  return ok;
}

// One pass: classify cur[0..cur_n) with pred (true = new side; `each` sees every point), then sum the new side's
// terms in order.  Leaves chain[0..nchains) and new_size in S.  SOLO: executed by warp 0 only.
// Chunks of (group size * kPiece) points: a thread owns a contiguous piece of each chunk so that the order survives.
// Returns true when the new side is the same set of points as in the previous pass (prev_masks, updated).
template <int THREADS, bool SOLO, typename Pred, typename Each>
__device__ __forceinline__ bool pass_sums(Shared &S, const Points &P, int cur_n, int nchains, unsigned *prev_masks, Pred pred,
                                          Each each) {
  const int tid = threadIdx.x;
  const int gsize = SOLO ? 32 : THREADS;
  const int chunk = gsize * kPiece;
  double acc = 0.0;
  int new_total = 0;
  bool same = true;
  int ci = 0;
  for (int base = 0; base < cur_n; base += chunk, ++ci) {
    const int n_here = min(chunk, cur_n - base);
    const int per = (n_here + gsize - 1) / gsize;  // <= kPiece
    const int lo = base + min(tid * per, n_here), hi = base + min(tid * per + per, n_here);
    // four points at a time: their index and colour loads are issued together (L2 round trips in the global mode)
    unsigned mask = 0;
    for (int j0 = lo; j0 < hi; j0 += 4) {
      int idx[4];
      uint32_t col[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) idx[q] = (j0 + q < hi) ? load_cur(P, j0 + q) : 0;
#pragma unroll
      for (int q = 0; q < 4; ++q) col[q] = (j0 + q < hi) ? P.colour[idx[q]] : 0u;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (j0 + q < hi) {
          const bool is_new = pred(col[q]);
          each(idx[q], is_new);
          mask |= (unsigned)is_new << (j0 + q - lo);
        }
      }
    }
    const bool changed = (mask != prev_masks[ci]);
    prev_masks[ci] = mask;
    int first, total;
    bool any_changed;
    group_ranks<THREADS, SOLO>(S, __popc(mask), changed, first, total, any_changed);
    same = same && !any_changed;
    bool summed = false;
    if (!SOLO && P.in_global && total >= kParMinTerms) summed = chunk_sums_parallel<THREADS>(S, P, lo, hi, mask, nchains, acc);
    for (int tile = 0; !summed && tile < total; tile += kTile) {
      // my new-side points have ranks [first, first + mine): stage those that fall into this tile
      int rank = first;
      for (int j0 = lo; j0 < hi; j0 += 4) {
        int idx[4];
        double wt[4];
        uint32_t col[4];
        bool take[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          take[q] = (j0 + q < hi) && ((mask >> (j0 + q - lo)) & 1u);
          idx[q] = take[q] ? load_cur(P, j0 + q) : 0;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          wt[q] = take[q] ? P.w[idx[q]] : 0.0;
          col[q] = take[q] ? P.colour[idx[q]] : 0u;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (take[q]) {
            if (rank >= tile && rank < tile + kTile) store_terms(S, rank - tile, wt[q], col[q], nchains);
            ++rank;
          }
        }
      }
      group_sync<SOLO>();
      add_terms(S, min(total - tile, kTile), nchains, acc);
      group_sync<SOLO>();
    }
    new_total += total;
  }
  if (tid < nchains) S.chain[tid] = acc;
  if (tid == 0) S.new_size = new_total;
  group_sync<SOLO>();
  return same;
}

// new centre from the chains, old centre by the 'combined mean' (:561-581, :780-810); lanes 0..2 = channels
template <bool SOLO>
__device__ __forceinline__ void derive_centres(Shared &S, bool with_squares) {
  const int t = threadIdx.x;
  if (t < 3) {
    const double nw = S.chain[3], ow = fsub(S.tw, nw);
    const double nm = fdiv(S.chain[t], nw);
    S.nm[t] = nm;
    S.om[t] = fdiv(fsub(fmul(S.tw, S.tm[t]), fmul(nw, nm)), ow);
    if (with_squares) S.nv[t] = S.chain[4 + t];
    if (t == 0) S.nw = nw, S.ow = ow;
  }
  group_sync<SOLO>();
}

// lhs / rhs of the hyperplane test (:616-623)
template <bool SOLO>
__device__ __forceinline__ void derive_hyperplane(Shared &S) {
  if (threadIdx.x == 0) {
    double l = fsub(fsq(S.om[0]), fsq(S.nm[0]));
    l = fadd(l, fsq(S.om[1]));
    l = fsub(l, fsq(S.nm[1]));
    l = fadd(l, fsq(S.om[2]));
    l = fsub(l, fsq(S.nm[2]));
    S.lhs = fmul(0.5, l);
    for (int c = 0; c < 3; ++c) S.rr[c] = fsub(S.om[c], S.nm[c]);
  }
  group_sync<SOLO>();
}

// split pass + max_iters LKM passes of one split (:438-811)
// prev_masks[kMaxChunks] is the caller's: on return it holds the membership masks of the last pass (bit q of chunk ci
// = this thread's q-th point of that chunk is on the new side).  mark_members: also write P.member (single-CTA form).
template <int THREADS, bool SOLO>
__device__ __forceinline__ void split_passes(Shared &S, const Points &P, int cur_n, int max_iters, int new_index, int old_index,
                                             unsigned *prev_masks, bool mark_members) {
#pragma unroll
  for (int i = 0; i < kMaxChunks; ++i) prev_masks[i] = 0xFFFFFFFFu;  // a piece has at most 16 points: never a real mask
  {
    const int axis = S.axis;
    const double cut = S.cut;
    pass_sums<THREADS, SOLO>(S, P, cur_n, 4, prev_masks, [&](uint32_t p) { return cut < chan(p, axis); }, [](int, bool) {});
  }
  derive_centres<SOLO>(S, false);
  for (int it = 0; it < max_iters; ++it) {
    derive_hyperplane<SOLO>(S);
    const double lhs = S.lhs, r0 = S.rr[0], r1 = S.rr[1], r2 = S.rr[2];
    const bool last = (it == max_iters - 1);
    const bool fixed_point = pass_sums<THREADS, SOLO>(
        S, P, cur_n, last ? 7 : 4, prev_masks,
        [&](uint32_t p) {
          const double dot = fadd(fadd(fmul(r0, chan(p, 0)), fmul(r1, chan(p, 1))), fmul(r2, chan(p, 2)));
          return !(lhs < dot);  // (:683)
        },
        [&](int idx, bool is_new) {
          if (last && mark_members) P.member[idx] = (uint16_t)(is_new ? new_index : old_index);
        });
    derive_centres<SOLO>(S, last);
    // Same new side as in the previous pass: the same sums, hence the same centres and the same side again, until
    // the last iteration -- which is the only one left to run (it also sums w*c*c and writes member[]).
    if (fixed_point && it < max_iters - 2) it = max_iters - 2;
  }
}

// Where the prologue finds the U points, through three arrays (colours, counts, first) whose meaning the source gives.
// FromTable: the histogram of a call -- colours = the unique colours in arrival order, counts = the direct count table
// (zeroed on the way), first = the first-seen table indexed by colour; the points are also left in A.pts[0].
struct FromTable {
  static __device__ __forceinline__ uint32_t colour(const uint32_t *uniq, int i) { return uniq[i]; }
  static __device__ __forceinline__ uint32_t first(const uint32_t *first_seen, int, uint32_t c) { return ld_cg_u32(first_seen + c); }
  static __device__ __forceinline__ uint32_t take_count(uint32_t *table, int, uint32_t c) {
    const uint32_t count = table[c];
    table[c] = 0u;  // the count table is all-zero again when the call ends
    return count;
  }
  static __device__ __forceinline__ void keep(const SplitArgs &A, int i, uint32_t c, uint32_t count) { A.pts[0][i] = make_uint2(c, count); }
};
// FromSlices: one item of a batch (dq_batch.cu) -- point i is (colours[i], counts[i]), first seen at pixel first[i].
struct FromSlices {
  static __device__ __forceinline__ uint32_t colour(const uint32_t *colours, int i) { return colours[i]; }
  static __device__ __forceinline__ uint32_t first(const uint32_t *first, int i, uint32_t) { return first[i]; }
  static __device__ __forceinline__ uint32_t take_count(uint32_t *counts, int i, uint32_t) { return counts[i]; }
  static __device__ __forceinline__ void keep(const SplitArgs &, int, uint32_t, uint32_t) {}
};

// The whole divisive phase of one input by one CTA of THREADS threads.  smem: sizeof(Shared) bytes; scratch:
// kScratchBytes of global memory (used when U > kSmemPoints).
// colours / counts / first: the points, read through Src (FromTable: the histogram and the first-seen table of the call);
// g_*: per-cluster scratch in global memory, used when K > kSmemColors.
template <int THREADS, typename Src = FromTable>
__device__ __noinline__ void split_exact_body(const SplitArgs &A, int U, unsigned char *smem, unsigned char *scratch, const uint32_t *colours,
                                 uint32_t *counts, const uint32_t *first, double *g_weight, double *g_tse, double *g_mean,
                                 double *g_var, int32_t *g_size) {
  Shared &S = *reinterpret_cast<Shared *>(smem);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int K = (int)A.num_colors;
  const bool in_smem = K <= kSmemColors;
  double *const weight = in_smem ? S.k_weight : g_weight;
  double *const tse = in_smem ? S.k_tse : g_tse;
  double *const mean = in_smem ? S.k_mean : g_mean;
  double *const var = in_smem ? S.k_var : g_var;
  int32_t *const size = in_smem ? S.k_size : g_size;
  Points P;
  if (U <= kSmemPoints) {
    P.keys = S.keys, P.w = S.w, P.colour = S.colour, P.member = S.member, P.cur = S.cur;
    P.cur_shared_across_ctas = false;
    P.in_global = false;
  } else {
    P.keys = reinterpret_cast<unsigned long long *>(scratch);
    P.w = reinterpret_cast<double *>(scratch + (size_t)kExactMaxPoints * 8);
    P.colour = reinterpret_cast<uint32_t *>(scratch + (size_t)kExactMaxPoints * 16);
    P.cur = reinterpret_cast<uint32_t *>(scratch + (size_t)kExactMaxPoints * 20);
    P.member = reinterpret_cast<uint16_t *>(scratch + (size_t)kExactMaxPoints * 28);
    P.cur_shared_across_ctas = false;
    P.in_global = true;
  }

  // ---- points in calc_color_table's emission order: (bucket asc, first seen desc) ----
  int sort_n = 32;
  while (sort_n < U) sort_n <<= 1;  // padding keys are all-ones: sorting the first power of two >= U is enough
  for (int i = tid; i < sort_n; i += THREADS) {
    unsigned long long key = ~0ull;
    if (i < U) {
      const uint32_t c = Src::colour(colours, i);
      const long R = (c >> 16) & 0xFF, G = (c >> 8) & 0xFF, B = c & 0xFF;
      const unsigned long long bucket = (unsigned long long)(((R * 33023 + G * 30013 + B * 27011) & 0x7fffffff) % 20023);
      key = (bucket << (31 + kIndexBits)) | ((unsigned long long)(0x7FFFFFFFu - Src::first(first, i, c)) << kIndexBits) |
            (unsigned long long)i;
    }
    P.keys[i] = key;
  }
  __syncthreads();
  for (int k = 2; k <= sort_n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < sort_n; i += THREADS) {
        const int partner = i ^ j;
        if (partner > i) {
          const unsigned long long a = P.keys[i], b = P.keys[partner];
          const bool up = (i & k) == 0;
          if ((a > b) == up) {
            P.keys[i] = b;
            P.keys[partner] = a;
          }
        }
      }
      __syncthreads();
    }
  }
  for (int i = tid; i < U; i += THREADS) {
    const int idx = (int)(P.keys[i] & ((1ull << kIndexBits) - 1ull));
    const uint32_t c = Src::colour(colours, idx);
    const uint32_t count = Src::take_count(counts, idx, c);
    P.colour[i] = c;
    P.w[i] = fmul(A.norm, (double)(int)count);  // weights[i] = weight * count (:185)
    P.member[i] = 0;
    P.cur[i] = (uint32_t)i;
    Src::keep(A, i, c, count);
  }
  for (int i = tid; i < K; i += THREADS) {  // `new T[n]()` of the reference (:296-324)
    weight[i] = 0.0;
    tse[i] = 0.0;
    size[i] = 0;
    for (int c = 0; c < 3; ++c) mean[3 * i + c] = 0.0, var[3 * i + c] = 0.0;
  }
  __syncthreads();  // keys are dead from here on: the union now holds terms

  // ---- DivQuantClusterInitMeanAndVar (:60-104): chains 0..2 mean, 4..6 second moments ----
  {
    unsigned no_prev[kMaxChunks];
#pragma unroll
    for (int i = 0; i < kMaxChunks; ++i) no_prev[i] = 0xFFFFFFFFu;
    pass_sums<THREADS, false>(S, P, U, 7, no_prev, [](uint32_t) { return true; }, [](int, bool) {});
  }
  if (tid == 0) {
    for (int c = 0; c < 3; ++c) {
      S.tm[c] = S.chain[c];
      S.tv[c] = fsub(S.chain[4 + c], fsq(S.chain[c]));
    }
    weight[0] = 1.0;
    size[0] = U;
    S.old_index = 0;
    S.cur_n = U;
  }
  __syncthreads();

  for (int new_index = 1; new_index < K; ++new_index) {
    const int old_index = S.old_index, cur_n = S.cur_n;
    if (tid == 0) {
      S.tw = weight[old_index];
      if (new_index > 1) {
        for (int c = 0; c < 3; ++c) S.tm[c] = mean[3 * old_index + c], S.tv[c] = var[3 * old_index + c];
      }
      int axis;
      double cut;
      choose_cut(S.tv, S.tm, axis, cut);
      S.axis = axis;
      S.cut = cut;
    }
    __syncthreads();
    {
      unsigned masks[kMaxChunks];
      if (cur_n <= kSolo) {
        if (warp == 0) split_passes<THREADS, true>(S, P, cur_n, A.max_iters, new_index, old_index, masks, true);
      } else {
        split_passes<THREADS, false>(S, P, cur_n, A.max_iters, new_index, old_index, masks, true);
      }
    }
    __syncthreads();

    if (tid == 0) {
      size[old_index] = cur_n - S.new_size;
      size[new_index] = S.new_size;
      for (int c = 0; c < 3; ++c) mean[3 * new_index + c] = S.nm[c], mean[3 * old_index + c] = S.om[c];
      SplitRecord r;
      if (A.records != nullptr) {
        r.new_index = new_index;
        r.old_index = old_index;
        r.cut_axis = S.axis;
        r.num_points = cur_n;
        r.new_size = S.new_size;
        r.is_last = (new_index == K - 1);
        r.cut_pos = S.cut;
        r.total_weight = S.tw;
        r.new_weight = S.nw;
        r.old_weight = S.ow;
        for (int c = 0; c < 3; ++c) {
          r.new_mean[c] = S.nm[c], r.old_mean[c] = S.om[c];
          r.new_var[c] = r.old_var[c] = 0.0;
        }
        r.new_tse = r.old_tse = 0.0;
      }
      if (new_index < K - 1) {  // the last split leaves without touching var / weight / tse (:823-832)
        double nv[3], ov[3];
        for (int c = 0; c < 3; ++c) {
          nv[c] = fsub(fdiv(S.nv[c], S.nw), fsq(S.nm[c]));  // (:836-838)
          ov[c] = fsub(fdiv(fsub(fmul(S.tw, S.tv[c]), fmul(S.nw, fadd(nv[c], fsq(fsub(S.nm[c], S.tm[c]))))), S.ow),
                       fsq(fsub(S.om[c], S.tm[c])));          // combined variance (:844-855)
          var[3 * new_index + c] = nv[c];
          var[3 * old_index + c] = ov[c];
        }
        weight[old_index] = S.ow;
        weight[new_index] = S.nw;
        tse[old_index] = fmul(S.ow, fadd(fadd(ov[0], ov[1]), ov[2]));  // (:871)
        tse[new_index] = fmul(S.nw, fadd(fadd(nv[0], nv[1]), nv[2]));
        if (A.records != nullptr) {
          for (int c = 0; c < 3; ++c) r.new_var[c] = nv[c], r.old_var[c] = ov[c];
          r.new_tse = tse[new_index];
          r.old_tse = tse[old_index];
        }
      }
      if (A.records != nullptr) A.records[new_index - 1] = r;
    }
    __syncthreads();
    if (new_index == K - 1) break;

    // ---- next cluster: strictly-greater scan seeded with DBL_MIN; stale old_index otherwise (:876-887) ----
    {
      double best = DBL_MIN;
      int best_i = -1;
      for (int ic = tid; ic <= new_index; ic += THREADS) {
        const double t = tse[ic];
        if (best < t) best = t, best_i = ic;
      }
      for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
        if (oi >= 0 && (best_i < 0 || best < ob || (ob == best && oi < best_i))) best = ob, best_i = oi;
      }
      if (lane == 0) S.red_val[warp] = best, S.red_idx[warp] = best_i;
      __syncthreads();
      if (tid == 0) {
        for (int q = 1; q < THREADS / 32; ++q) {
          const double ob = S.red_val[q];
          const int oi = S.red_idx[q];
          if (oi >= 0 && (best_i < 0 || best < ob || (ob == best && oi < best_i))) best = ob, best_i = oi;
        }
        if (best_i >= 0) S.old_index = best_i;
      }
      __syncthreads();
    }
    // ---- steady state: the split just made put every point on the old side, left the old cluster's statistics bit for bit
    //      as they were and the same cluster is up again -- so the next split starts from the very inputs this one had and
    //      every split that is left repeats it (K far above the number of colours: the tail of empty clusters, :876-887
    //      with no TSE above DBL_MIN).  The arg-max cannot change either: the only new entry of tse[] equals the one that did
    //      not win this time.  The remaining clusters are filled in instead of computed ----
    if (tid == 0) {
      bool steady = S.new_size == 0 && S.old_index == old_index;
      if (steady) {
        steady = same_input(weight[old_index], S.tw);
        for (int c = 0; c < 3; ++c)
          steady = steady && same_input(mean[3 * old_index + c], S.tm[c]) && same_input(var[3 * old_index + c], S.tv[c]);
      }
      S.steady = steady ? 1 : 0;
    }
    __syncthreads();
    if (S.steady) {
      for (int ni = new_index + 1 + tid; ni < K; ni += THREADS) {
        const bool last = (ni == K - 1);
        size[ni] = 0;
        for (int c = 0; c < 3; ++c) mean[3 * ni + c] = mean[3 * new_index + c];
        if (!last) {  // (the last split touches neither var nor weight nor tse, :823-832)
          for (int c = 0; c < 3; ++c) var[3 * ni + c] = var[3 * new_index + c];
          weight[ni] = weight[new_index];
          tse[ni] = tse[new_index];
        }
        if (A.records != nullptr) {
          SplitRecord r = A.records[new_index - 1];
          r.new_index = ni;
          r.is_last = last;
          if (last) {
            for (int c = 0; c < 3; ++c) r.new_var[c] = r.old_var[c] = 0.0;
            r.new_tse = r.old_tse = 0.0;
          }
          A.records[ni - 1] = r;
        }
      }
      __syncthreads();
      break;
    }
    // ---- gather its points in ascending original order (:929-1019): contiguous pieces + exclusive scan ----
    {
      const uint16_t want = (uint16_t)S.old_index;
      const int chunk = THREADS * kPiece;
      int written = 0;
      for (int base = 0; base < U; base += chunk) {
        const int n_here = min(chunk, U - base);
        const int per = (n_here + THREADS - 1) / THREADS;
        const int lo = base + min(tid * per, n_here), hi = base + min(tid * per + per, n_here);
        unsigned mask = 0;
        for (int i = lo; i < hi; ++i) mask |= (unsigned)(P.member[i] == want) << (i - lo);
        int first, total;
        bool unused;
        group_ranks<THREADS, false>(S, __popc(mask), false, first, total, unused);
        int pos = written + first;
        for (int i = lo; i < hi; ++i)
          if ((mask >> (i - lo)) & 1u) P.cur[pos++] = (uint32_t)i;
        written += total;
      }
      if (tid == 0) {
        S.cur_n = written;
        if (written != size[S.old_index]) A.ctl[kCtlError] = 7;  // "Cluster to be split is expected to be of size ..." (:1013)
      }
      __syncthreads();
    }
  }

  // ---- palette = rounded means of the non-empty clusters in index order (:1030-1065) ----
  if (tid == 0) S.emitted = 0;
  __syncthreads();
  for (int base = 0; base < K; base += THREADS) {
    const int ic = base + tid;
    uint32_t colour = 0;
    int sz = 0;
    if (ic < K) {
      sz = (K > 1) ? size[ic] : U;
      double m[3] = {0.0, 0.0, 0.0};  // K == 1 never assigns mean[0] (SURVEY 7 quirk)
      if (K > 1) m[0] = mean[3 * ic], m[1] = mean[3 * ic + 1], m[2] = mean[3 * ic + 2];
      if (sz > 0) {
        const uint32_t Rr = (__double2uint_rz(fadd(m[0], 0.5)) & 0xFFu) << A.shift;
        const uint32_t Gg = (__double2uint_rz(fadd(m[1], 0.5)) & 0xFFu) << A.shift;
        const uint32_t Bb = (__double2uint_rz(fadd(m[2], 0.5)) & 0xFFu) << A.shift;
        colour = (Rr << 16) | (Gg << 8) | Bb;
      }
      A.cluster_size[ic] = (uint32_t)sz;
      for (int c = 0; c < 3; ++c) A.cluster_mean[3 * ic + c] = m[c];
    }
    int first, total;
    bool unused;
    group_ranks<THREADS, false>(S, sz > 0 ? 1 : 0, false, first, total, unused);
    if (sz > 0) A.palette[S.emitted + first] = colour;
    __syncthreads();
    if (tid == 0) S.emitted += total;
    __syncthreads();
  }
  if (tid == 0) {
    A.result[0] = (uint32_t)S.emitted;
    A.result[1] = (uint32_t)(K - S.emitted);
    A.ctl[kCtlDone] = 1;
    A.ctl[kCtlRounds] = (uint32_t)(K - 1);
    A.ctl[kCtlSplits] = (uint32_t)(K - 1);
  }
}

}  // namespace exact

// first_seen pass shared by the fused and the stand-alone form: smallest sample index of every colour (sampling and bit
// cutting as in hist_insert, whose first toucher of every colour has set the entry to 0xFFFFFFFF).
__device__ __forceinline__ void exact_first_seen(const ExactSampling &q, uint32_t *first_seen, uint32_t thread, uint32_t threads) {
  for (uint32_t s = thread; s < q.num_samples; s += threads) {
    const uint32_t ir = (s / q.samples_per_row) * q.dec, ic = (s % q.samples_per_row) * q.dec;
    // the reference's addressing, bug included (MapColors.cpp:120-122)
    const uint32_t c = (q.in[ic + ir * q.num_rows] & q.word_mask) >> q.shift;
    if (s < first_seen[c]) atomicMin(first_seen + c, s);  // the plain read only skips atomics that cannot win
  }
}

}  // namespace dq

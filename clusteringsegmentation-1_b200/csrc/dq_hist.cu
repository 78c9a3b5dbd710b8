// dq_hist.cu -- 24-bit colour histogram / unique-colour extraction.
//
// Reference: calc_color_table, DivQuant/DivQuantMapColors.cpp:82-203 (20 023-bucket chained hash),
// and the cut_bits pre-quantisation it is fed with, DivQuant/DivQuantUni.cpp:28-100.
//
// Device formulation: 24-bit colours are a perfect hash of themselves, so the "global hash" is a
// direct-addressed table of 2^24 u32 counters (64 MB of the 180 GB HBM; only the sectors of colours
// that occur are ever touched, so for natural images the working set lives in L2).  The table is
// all-zero between calls: whoever dirties it clears exactly the entries it touched.
//   hist_insert   : count += 1 per sampled pixel; the thread that sees 0 appends the colour to the
//                   unique list (one warp-aggregated cursor bump per warp).  Contiguous inputs of a 32 768-pixel
//                   chunk per SM or more are counted per chunk in shared memory first (dq_hist_chunk.cuh).
//   hist_collect  : (colour, count) points for the divisive phase.
//   table_clear   : zero the touched entries.
#include <mutex>
#include <set>

#include "dq_hist_chunk.cuh"
#include "dq_kernels.cuh"

namespace dq {
namespace {

// Contiguous sampling (dec_factor == 1, numRows == 1: every live caller, quant_util.cpp:60).
__global__ void __launch_bounds__(256) hist_insert_kernel(const uint32_t *__restrict__ in, uint32_t n,
                                                         uint32_t word_mask, uint32_t shift, uint32_t *table,
                                                         uint32_t *uniq, uint32_t *ucount, uint32_t *seen_init) {
  const uint32_t nvec = n >> 2;
  const uint4 *in4 = reinterpret_cast<const uint4 *>(in);
  const uint32_t stride = gridDim.x * blockDim.x;
  // whole warps iterate together so the ballots inside insert_colour are convergent
  const uint32_t nvec_round = (nvec + 31u) & ~31u;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nvec_round; i += stride) {
    const bool ok = i < nvec;
    uint4 p = make_uint4(0, 0, 0, 0);
    if (ok) p = __ldcs(in4 + i);  // streamed once: keep L2 for the table
    // all four atomics are issued before any of their results is looked at (4 L2 round trips in flight)
    const uint32_t c[4] = {cut_colour(p.x, word_mask, shift), cut_colour(p.y, word_mask, shift),
                           cut_colour(p.z, word_mask, shift), cut_colour(p.w, word_mask, shift)};
    uint32_t old[4] = {1u, 1u, 1u, 1u};
    if (ok) {
#pragma unroll
      for (int k = 0; k < 4; ++k) old[k] = atomicAdd(table + c[k], 1u);
    }
    // a thread's own duplicates: only the first one can have seen 0, nothing to fix up
    unsigned m[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) m[k] = __ballot_sync(0xffffffffu, old[k] == 0u);
    const unsigned any = m[0] | m[1] | m[2] | m[3];
    if (any) {
      const int lane = threadIdx.x & 31;
      const uint32_t total = __popc(m[0]) + __popc(m[1]) + __popc(m[2]) + __popc(m[3]);
      uint32_t base = 0;
      if (lane == 0) base = atomicAdd(ucount, total);
      base = __shfl_sync(0xffffffffu, base, 0);
      const unsigned below = (1u << lane) - 1u;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (old[k] == 0u) {
          uniq[base + __popc(m[k] & below)] = c[k];
          if (seen_init) seen_init[c[k]] = 0xFFFFFFFFu;
        }
        base += __popc(m[k]);
      }
    }
  }
  // tail (< 4 pixels) handled by the first warp of the grid
  if (blockIdx.x == 0 && threadIdx.x < 32) {
    const uint32_t i = (nvec << 2) + threadIdx.x;
    const bool ok = i < n;
    const uint32_t p = ok ? in[i] : 0u;
    insert_colour(cut_colour(p, word_mask, shift), ok, table, uniq, ucount, seen_init);
  }
}

// General sampling grid of calc_color_table (:120-124), including its `ic + ir*numRows` addressing.
__global__ void __launch_bounds__(256) hist_insert_sampled_kernel(const uint32_t *__restrict__ in, uint32_t samples_per_row,
                                                                 uint32_t num_samples, uint32_t num_rows, uint32_t dec,
                                                                 uint32_t word_mask, uint32_t shift, uint32_t *table,
                                                                 uint32_t *uniq, uint32_t *ucount, uint32_t *seen_init) {
  const uint32_t stride = gridDim.x * blockDim.x;
  const uint32_t round = (num_samples + 31u) & ~31u;
  for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < round; s += stride) {
    const bool ok = s < num_samples;
    uint32_t p = 0;
    if (ok) {
      const uint32_t ir = (s / samples_per_row) * dec, ic = (s % samples_per_row) * dec;
      p = in[ic + ir * num_rows];
    }
    insert_colour(cut_colour(p, word_mask, shift), ok, table, uniq, ucount, seen_init);
  }
}

// (colour, count) points for the divisive phase.  With `clear` the counter is zeroed on the way out, which
// restores the count table's all-zero invariant without a separate pass.
__global__ void __launch_bounds__(256) hist_collect_kernel(const uint32_t *__restrict__ uniq, const uint32_t *ucount,
                                                          uint32_t *table, uint2 *pts, int clear) {
  const uint32_t u = *ucount;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < u; i += gridDim.x * blockDim.x) {
    const uint32_t c = uniq[i];
    pts[i] = make_uint2(c, table[c]);
    if (clear) table[c] = 0u;
  }
}

__global__ void __launch_bounds__(256) table_clear_kernel(const uint32_t *__restrict__ uniq, const uint32_t *ucount,
                                                         uint32_t *table) {
  const uint32_t u = *ucount;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < u; i += gridDim.x * blockDim.x) table[uniq[i]] = 0u;
}

// allPixelsUnique path: every pixel is a point of weight 1 (DivQuantCluster.cpp:1130-1132).
__global__ void __launch_bounds__(256) points_from_pixels_kernel(const uint32_t *__restrict__ in, uint32_t n, uint2 *pts) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    pts[i] = make_uint2(in[i] & 0x00FFFFFFu, 1u);
}

// cut_bits proper (DivQuantUni.cpp:60-91), for the stand-alone entry point.
__global__ void __launch_bounds__(256) cut_bits_kernel(const uint32_t *__restrict__ in, uint32_t n, uint32_t *out,
                                                      uint32_t sr, uint32_t sg, uint32_t sb) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t p = in[i];
    if (sr == sg && sr == sb) {
      const uint32_t byte_mask = (0xFFu >> sr) << sr;
      out[i] = (p & ((byte_mask << 16) | (byte_mask << 8) | byte_mask)) >> sr;
    } else {
      out[i] = ((((p >> 16) & 0xFFu) >> sr) << 16) | ((((p >> 8) & 0xFFu) >> sg) << 8) | ((p & 0xFFu) >> sb);
    }
  }
}

// First sampled position of every unique colour (needed only to reproduce calc_color_table's
// emission order): table[c] = min(sample index).  Entries must hold 0xFFFFFFFF on entry.
__global__ void __launch_bounds__(256) first_seen_kernel(const uint32_t *__restrict__ in, uint32_t samples_per_row,
                                                        uint32_t num_samples, uint32_t num_rows, uint32_t dec,
                                                        uint32_t word_mask, uint32_t shift, uint32_t *table) {
  for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < num_samples; s += gridDim.x * blockDim.x) {
    const uint32_t ir = (s / samples_per_row) * dec, ic = (s % samples_per_row) * dec;
    atomicMin(table + cut_colour(in[ic + ir * num_rows], word_mask, shift), s);
  }
}

__global__ void __launch_bounds__(256) table_fill_kernel(const uint32_t *__restrict__ uniq, uint32_t u, uint32_t *table,
                                                        uint32_t value) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < u; i += gridDim.x * blockDim.x) table[uniq[i]] = value;
}

// (bucket, first-seen) sort keys: ascending key order == the reference's emission order, i.e. bucket
// ascending and, inside a bucket, most recently first-seen colour first (:157-158, :174-198).
__global__ void __launch_bounds__(256) order_keys_kernel(const uint2 *__restrict__ pts, uint32_t u, const uint32_t *table,
                                                        uint64_t *keys) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < u; i += gridDim.x * blockDim.x) {
    const uint32_t c = pts[i].x;
    const long R = (c >> 16) & 0xFF, G = (c >> 8) & 0xFF, B = c & 0xFF;
    const uint32_t bucket = (uint32_t)(((R * 33023 + G * 30013 + B * 27011) & 0x7fffffff) % 20023);  // HASH (:59-62)
    keys[i] = ((uint64_t)bucket << 32) | (uint64_t)(0xFFFFFFFFu - table[c]);
  }
}

// ---- emission order on the device: bitonic sort of the (unique) keys with the point index as payload, then the
//      unique colours and their weights count * (1/N) written out in that order (calc_color_table :172-198) ----
__global__ void __launch_bounds__(256) order_pad_kernel(uint64_t *keys, uint32_t *vals, uint32_t u, uint32_t n_pow2) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pow2; i += gridDim.x * blockDim.x) {
    vals[i] = i;
    if (i >= u) keys[i] = ~0ull;  // padding sorts to the end
  }
}
__global__ void __launch_bounds__(256) bitonic_step_kernel(uint64_t *keys, uint32_t *vals, uint32_t n_pow2, uint32_t j, uint32_t k) {
  const uint32_t half = n_pow2 >> 1;
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < half; p += gridDim.x * blockDim.x) {
    const uint32_t i = ((p & ~(j - 1u)) << 1) | (p & (j - 1u));  // the p-th index whose bit j is clear
    const uint64_t a = keys[i], b = keys[i | j];
    if ((a > b) == ((i & k) == 0u)) {
      keys[i] = b;
      keys[i | j] = a;
      const uint32_t va = vals[i];
      vals[i] = vals[i | j];
      vals[i | j] = va;
    }
  }
}
__global__ void __launch_bounds__(256) order_emit_kernel(const uint2 *__restrict__ pts, const uint32_t *__restrict__ vals, uint32_t u,
                                                        double norm, uint32_t *colours, double *weights) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < u; i += gridDim.x * blockDim.x) {
    const uint2 p = pts[vals[i]];
    colours[i] = p.x;
    weights[i] = __dmul_rn(norm, (double)(int)p.y);  // weights[i] = norm_factor * bucket->value (:185), value is an int
  }
}

// Same into a fixed-capacity slice of the exchange buffers: entries beyond the shard's U get count 0 (the merge skips
// them), a shard with more than `cap` colours raises *overflow (the caller sized the exchange too small).
// With `first` (cap + 1 words): first[i] = the shard-local first-seen index of colour i (read from first_table), and
// first[cap] = the shard's pixel count, from which the merge derives every shard's offset in the whole image.
__global__ void __launch_bounds__(256) hist_export_padded_kernel(const uint2 *__restrict__ pts, const uint32_t *ucount, uint32_t cap,
                                                                uint32_t *colours, uint32_t *counts, uint32_t *overflow,
                                                                const uint32_t *__restrict__ first_table, uint32_t *first,
                                                                uint32_t n_shard) {
  const uint32_t u = *ucount;
  if (u > cap && blockIdx.x == 0 && threadIdx.x == 0) *overflow = u;
  if (first && blockIdx.x == 0 && threadIdx.x == 0) first[cap] = n_shard;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += gridDim.x * blockDim.x) {
    if (i < u) {
      const uint2 p = pts[i];
      colours[i] = p.x;
      counts[i] = p.y;
      if (first) first[i] = first_table[p.x];
    } else {
      counts[i] = 0u;
    }
  }
}

// Merge of gathered per-shard lists into the direct table: counts add up exactly; the entry that bumps a
// counter from 0 appends the colour to the merged unique list (and, with seen_init, sets its first-seen entry to
// 0xFFFFFFFF for hist_merge_first_kernel, as hist_insert does for the first-seen pass over pixels).
__global__ void __launch_bounds__(256) hist_merge_kernel(const uint32_t *__restrict__ colours, const uint32_t *__restrict__ counts,
                                                        uint32_t n, uint32_t *table, uint32_t *uniq, uint32_t *ucount,
                                                        uint32_t *seen_init) {
  const uint32_t stride = gridDim.x * blockDim.x;
  const uint32_t round = (n + 31u) & ~31u;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < round; i += stride) {
    const bool ok = i < n && counts[i] != 0;
    const uint32_t c = ok ? (colours[i] & 0x00FFFFFFu) : 0u;
    bool fresh = false;
    if (ok) fresh = (atomicAdd(table + c, counts[i]) == 0u);
    const unsigned m = __ballot_sync(0xffffffffu, fresh);
    if (m) {
      const int lane = threadIdx.x & 31;
      uint32_t base = 0;
      if (lane == __ffs(m) - 1) base = atomicAdd(ucount, (uint32_t)__popc(m));
      base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
      if (fresh) {
        uniq[base + __popc(m & ((1u << lane) - 1u))] = c;
        if (seen_init) seen_init[c] = 0xFFFFFFFFu;
      }
    }
  }
}

// First-seen index of every colour over the whole image from the gathered lists: shard w's rows start at the sum of the
// pixel counts of shards 0..w-1 (rows are contiguous and in rank order), so the image's index of a colour is the minimum
// over shards of (offset + shard-local index).  colours / counts: [world][cap], first: [world][cap + 1].
__global__ void __launch_bounds__(256) hist_merge_first_kernel(const uint32_t *__restrict__ colours, const uint32_t *__restrict__ counts,
                                                              const uint32_t *__restrict__ first, uint32_t cap, uint32_t world,
                                                              uint32_t *first_seen) {
  const uint32_t n = world * cap;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (counts[i] == 0u) continue;
    const uint32_t w = i / cap;
    uint32_t offset = 0;
    for (uint32_t v = 0; v < w; ++v) offset += first[v * (cap + 1) + cap];
    atomicMin(first_seen + (colours[i] & 0x00FFFFFFu), offset + first[w * (cap + 1) + (i - w * cap)]);
  }
}

// hist_insert_chunked_kernel's table is above the default 48 KB of dynamic shared memory: the limit is raised once per device.
void hist_chunk_allow_smem() {
  static std::mutex mu;
  static std::set<int> raised;
  int dev = 0;
  DQ_CUDA_CHECK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  if (raised.insert(dev).second)
    DQ_CUDA_CHECK(cudaFuncSetAttribute(hist_insert_chunked_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hist_chunk::kSmemBytes));
}

inline int blocks_for(uint64_t items, int threads, int sm_count, int per_sm) {
  uint64_t want = (items + threads - 1) / threads;
  uint64_t cap = (uint64_t)sm_count * per_sm;
  if (want < 1) want = 1;
  return (int)(want < cap ? want : cap);
}

}  // namespace

void hist_insert(const uint32_t *d_in, uint32_t n, uint32_t num_rows, uint32_t num_cols, uint32_t dec, int num_bits,
                 uint32_t *d_table, uint32_t *d_uniq, uint32_t *d_ucount, int sm_count, cudaStream_t st, uint32_t *d_seen_init) {
  const uint32_t shift = 8u - (uint32_t)num_bits;
  const uint32_t byte_mask = (0xFFu >> shift) << shift;
  const uint32_t word_mask = (byte_mask << 16) | (byte_mask << 8) | byte_mask;
  const bool aligned = (reinterpret_cast<uintptr_t>(d_in) & 15u) == 0;  // uint4 loads
  if (dec == 1 && num_rows == 1 && aligned) {
    const uint32_t count = num_cols < n ? num_cols : n;
    if (count / hist_chunk::kChunk >= (uint32_t)sm_count) {
      // a chunk per SM or more (4K frames): one L2 atomic per distinct colour of a chunk instead of one per pixel
      hist_chunk_allow_smem();
      hist_insert_chunked_kernel<<<blocks_for(count, (int)hist_chunk::kChunk, sm_count, 8), hist_chunk::kThreads,
                                   hist_chunk::kSmemBytes, st>>>(d_in, count, hist_chunk::kChunk >> 2, word_mask, shift,
                                                                 d_table, d_uniq, d_ucount, d_seen_init);
    } else {
      hist_insert_kernel<<<blocks_for((count >> 2) + 32, 256, sm_count, 8), 256, 0, st>>>(d_in, count, word_mask, shift,
                                                                                          d_table, d_uniq, d_ucount, d_seen_init);
    }
  } else {
    const uint32_t nr = (num_rows + dec - 1) / dec, nc = (num_cols + dec - 1) / dec;
    const uint32_t samples = nr * nc;
    hist_insert_sampled_kernel<<<blocks_for(samples, 256, sm_count, 8), 256, 0, st>>>(d_in, nc, samples, num_rows, dec,
                                                                                     word_mask, shift, d_table, d_uniq,
                                                                                     d_ucount, d_seen_init);
  }
  DQ_CUDA_CHECK(cudaGetLastError());
}

void hist_collect(const uint32_t *d_uniq, const uint32_t *d_ucount, uint32_t u_hint, uint32_t *d_table, uint2 *d_pts,
                  bool clear_table, int sm_count, cudaStream_t st) {
  hist_collect_kernel<<<blocks_for(u_hint, 256, sm_count, 8), 256, 0, st>>>(d_uniq, d_ucount, d_table, d_pts, clear_table ? 1 : 0);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void table_clear(const uint32_t *d_uniq, const uint32_t *d_ucount, uint32_t u_hint, uint32_t *d_table, int sm_count,
                 cudaStream_t st) {
  table_clear_kernel<<<blocks_for(u_hint, 256, sm_count, 8), 256, 0, st>>>(d_uniq, d_ucount, d_table);
  DQ_CUDA_CHECK(cudaGetLastError());
}

// Sorts d_keys[0..u) ascending with d_vals = the index each key came from (both arrays hold the power of two >= u entries).
void order_sort(uint64_t *d_keys, uint32_t *d_vals, uint32_t u, int sm_count, cudaStream_t st) {
  if (u == 0) return;
  uint32_t n_pow2 = 2;
  while (n_pow2 < u) n_pow2 <<= 1;
  order_pad_kernel<<<blocks_for(n_pow2, 256, sm_count, 8), 256, 0, st>>>(d_keys, d_vals, u, n_pow2);
  for (uint32_t k = 2; k <= n_pow2; k <<= 1)
    for (uint32_t j = k >> 1; j > 0; j >>= 1)
      bitonic_step_kernel<<<blocks_for(n_pow2 >> 1, 256, sm_count, 8), 256, 0, st>>>(d_keys, d_vals, n_pow2, j, k);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void order_sort_emit(const uint2 *d_pts, uint32_t u, uint64_t *d_keys, uint32_t *d_vals, double norm, uint32_t *d_colours,
                     double *d_weights, int sm_count, cudaStream_t st) {
  if (u == 0) return;
  order_sort(d_keys, d_vals, u, sm_count, st);
  order_emit_kernel<<<blocks_for(u, 256, sm_count, 8), 256, 0, st>>>(d_pts, d_vals, u, norm, d_colours, d_weights);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void hist_export_padded(const uint2 *d_pts, const uint32_t *d_ucount, uint32_t cap, uint32_t *d_colours, uint32_t *d_counts,
                        uint32_t *d_overflow, int sm_count, cudaStream_t st, const uint32_t *d_first_table, uint32_t *d_first,
                        uint32_t n_shard) {
  hist_export_padded_kernel<<<blocks_for(cap, 256, sm_count, 8), 256, 0, st>>>(d_pts, d_ucount, cap, d_colours, d_counts, d_overflow,
                                                                              d_first_table, d_first, n_shard);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void hist_merge(const uint32_t *d_colours, const uint32_t *d_counts, uint32_t num_entries, uint32_t *d_table, uint32_t *d_uniq,
                uint32_t *d_ucount, int sm_count, cudaStream_t st, uint32_t *d_seen_init) {
  hist_merge_kernel<<<blocks_for(num_entries, 256, sm_count, 8), 256, 0, st>>>(d_colours, d_counts, num_entries, d_table, d_uniq,
                                                                               d_ucount, d_seen_init);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void hist_merge_first(const uint32_t *d_colours, const uint32_t *d_counts, const uint32_t *d_first, uint32_t cap, uint32_t world,
                      uint32_t *d_first_seen, int sm_count, cudaStream_t st) {
  hist_merge_first_kernel<<<blocks_for((uint64_t)world * cap, 256, sm_count, 8), 256, 0, st>>>(d_colours, d_counts, d_first, cap, world,
                                                                                             d_first_seen);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void points_from_pixels(const uint32_t *d_in, uint32_t n, uint2 *d_pts, int sm_count, cudaStream_t st) {
  points_from_pixels_kernel<<<blocks_for(n, 256, sm_count, 8), 256, 0, st>>>(d_in, n, d_pts);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void cut_bits_device(const uint32_t *d_in, uint32_t n, uint32_t *d_out, int rbits, int gbits, int bbits, int sm_count,
                     cudaStream_t st) {
  cut_bits_kernel<<<blocks_for(n, 256, sm_count, 8), 256, 0, st>>>(d_in, n, d_out, 8u - rbits, 8u - gbits, 8u - bbits);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void order_keys(const uint32_t *d_in, uint32_t num_rows, uint32_t num_cols, uint32_t dec, int num_bits, const uint32_t *d_uniq,
                const uint2 *d_pts, uint32_t u, uint32_t *d_table, uint64_t *d_keys, int sm_count, cudaStream_t st) {
  const uint32_t shift = 8u - (uint32_t)num_bits;
  const uint32_t byte_mask = (0xFFu >> shift) << shift;
  const uint32_t word_mask = (byte_mask << 16) | (byte_mask << 8) | byte_mask;
  const uint32_t nr = (num_rows + dec - 1) / dec, nc = (num_cols + dec - 1) / dec;
  const uint32_t samples = nr * nc;
  table_fill_kernel<<<blocks_for(u, 256, sm_count, 8), 256, 0, st>>>(d_uniq, u, d_table, 0xFFFFFFFFu);
  first_seen_kernel<<<blocks_for(samples, 256, sm_count, 8), 256, 0, st>>>(d_in, nc, samples, num_rows, dec, word_mask,
                                                                          shift, d_table);
  order_keys_kernel<<<blocks_for(u, 256, sm_count, 8), 256, 0, st>>>(d_pts, u, d_table, d_keys);
  table_fill_kernel<<<blocks_for(u, 256, sm_count, 8), 256, 0, st>>>(d_uniq, u, d_table, 0u);
  DQ_CUDA_CHECK(cudaGetLastError());
}

}  // namespace dq

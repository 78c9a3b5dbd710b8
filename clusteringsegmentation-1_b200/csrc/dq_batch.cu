// dq_batch.cu -- quant_recurse over many small independent pixel sets ("items") in a few launches.
//
// An item that fits the ordered path in shared memory (at most kBatchMaxPoints distinct colours, K <= 512) runs the same
// arithmetic as its single call on that path (dq_split_exact.cuh): what changes is only where the points come from and
// that one CTA per item works next to the others instead of one call holding the whole GPU.
//   batch_hist_kernel    one CTA per item: unique colours, counts and first-seen pixel index in a shared-memory hash
//                        table (not the 2^24 direct table); more than kBatchMaxPoints colours marks the item for the
//                        single-call path
//   batch_split_kernel   one CTA per item: split_exact_body on the item's (colour, count, first-seen) slices
//   (host)               palettes back in one copy; the reference's duplicate removal, std::sort and lut_init per item
//                        (dq_context.cu), tables up in one copy
//   batch_remap_kernel   one CTA per tile of an item's pixels: the keyed integer arg-min of dq_map_int.cuh
#include "dq_kernels.cuh"
#include "dq_map_int.cuh"
#include "dq_split_exact.cuh"

#include <algorithm>

namespace dq {
namespace {

constexpr int kBatchThreads = 256;
constexpr int kHashSlots = 2 * kBatchMaxPoints;  // load <= 1/2 while an item can still be batched
constexpr uint32_t kEmptySlot = 0xFFFFFFFFu;     // colours are 24-bit words: all-ones is free
static_assert((kHashSlots & (kHashSlots - 1)) == 0, "power-of-two table");
static_assert(kBatchMaxPoints <= (uint32_t)exact::kSmemPoints, "a batched item keeps its points in shared memory");
static_assert(kSplit2MaxColors <= (uint32_t)exact::kSmemColors && kSplit2MaxColors <= (uint32_t)kIntColors,
              "a batched item keeps its clusters and its palette in shared memory");
constexpr size_t kHistSmemBytes = (size_t)3 * kHashSlots * sizeof(uint32_t);

__global__ void __launch_bounds__(kBatchThreads) batch_hist_kernel(const uint32_t *__restrict__ in, const BatchItem *items,
                                                                    uint32_t *colours, uint32_t *counts, uint32_t *first,
                                                                    uint32_t *res) {
  extern __shared__ __align__(16) uint32_t hist_smem[];
  uint32_t *s_key = hist_smem, *s_cnt = hist_smem + kHashSlots, *s_first = hist_smem + 2 * kHashSlots;
  __shared__ uint32_t s_u, s_over, s_pos;
  const int tid = threadIdx.x;
  const BatchItem it = items[blockIdx.x];
  uint32_t *r = res + (size_t)blockIdx.x * kBatchResultWords;
  // the item's result and ctl words start at zero, as reset_control leaves them for a single call (the split sets the
  // error word only when something is wrong, and the buffer is reused from call to call)
  if (tid < (int)kBatchResultWords) r[tid] = 0u;
  for (int i = tid; i < kHashSlots; i += kBatchThreads) s_key[i] = kEmptySlot, s_cnt[i] = 0u, s_first[i] = 0xFFFFFFFFu;
  if (tid == 0) s_u = 0u, s_over = 0u, s_pos = 0u;
  __syncthreads();
  const uint32_t *px = in + it.begin;
  // Every thread claims at most one slot after the overflow flag is raised, so at most kBatchMaxPoints + kBatchThreads
  // slots are ever taken and every probe ends.
  for (uint32_t i = tid; i < it.n; i += kBatchThreads) {
    if (*(volatile uint32_t *)&s_over) break;
    const uint32_t c = px[i] & 0x00FFFFFFu;  // quant_recurse: 8 bits per channel, alpha ignored
    uint32_t h = (c * 2654435761u) >> 19;    // 13 bits
    for (;;) {
      const uint32_t k = *(volatile uint32_t *)&s_key[h];
      if (k == c) break;
      if (k == kEmptySlot) {
        const uint32_t prev = atomicCAS(&s_key[h], kEmptySlot, c);
        if (prev == kEmptySlot) {
          if (atomicAdd(&s_u, 1u) >= kBatchMaxPoints) s_over = 1u;
          break;
        }
        if (prev == c) break;
      }
      h = (h + 1u) & (kHashSlots - 1);
    }
    atomicAdd(&s_cnt[h], 1u);
    atomicMin(&s_first[h], i);  // the smallest index wins whatever order the threads come in
  }
  __syncthreads();
  if (s_over) {
    if (tid == 0) r[0] = kBatchOverflow;
    return;
  }
  // The order of the slices does not matter: the split sorts the points by (bucket, first seen), and no two colours
  // share a first-seen index.
  for (int i = tid; i < kHashSlots; i += kBatchThreads) {
    const uint32_t c = s_key[i];
    if (c == kEmptySlot) continue;
    const uint32_t pos = it.begin + atomicAdd(&s_pos, 1u);
    colours[pos] = c;
    counts[pos] = s_cnt[i];
    first[pos] = s_first[i];
  }
  if (tid == 0) r[0] = s_u;
}

// (one CTA per SM: sizeof(exact::Shared) of shared memory; the register budget that leaves keeps split_exact_body free of spills)
__global__ void __launch_bounds__(kBatchThreads, 1) batch_split_kernel(const BatchItem *items, uint32_t max_points, const uint32_t *colours,
                                                                     uint32_t *counts, const uint32_t *first, uint32_t *res,
                                                                     uint32_t *palette, uint32_t *cluster_size, double *cluster_mean) {
  extern __shared__ __align__(16) unsigned char batch_smem[];
  __shared__ SplitArgs s_args;
  const BatchItem it = items[blockIdx.x];
  uint32_t *r = res + (size_t)blockIdx.x * kBatchResultWords;
  const uint32_t U = r[0];
  if (U > max_points || U == 0u) return;  // (the single-call path takes it)
  if (threadIdx.x == 0) {
    SplitArgs a = {};
    a.num_points = U;
    a.num_colors = it.k;
    a.max_iters = 10;  // quant_recurse (quant_util.cpp:31)
    a.shift = 0;
    a.norm = fdiv(1.0, (double)it.n);  // sample_norm(1, n, 1) bit for bit: IEEE division
    a.ctl = r + 4;
    a.result = r + 1;
    a.palette = palette + it.pal;
    a.cluster_size = cluster_size + it.pal;
    a.cluster_mean = cluster_mean + 3 * (size_t)it.pal;
    s_args = a;
  }
  __syncthreads();
  exact::split_exact_body<kBatchThreads, exact::FromSlices>(s_args, (int)U, batch_smem, nullptr, colours + it.begin, counts + it.begin,
                                                            first + it.begin, nullptr, nullptr, nullptr, nullptr, nullptr);
}

constexpr int kRemapPix = kBatchTilePixels / kBatchThreads;  // pixels per thread and tile
static_assert(kBatchTilePixels % kBatchThreads == 0, "whole tiles");

// kLabels: also labels[p] = the caller's palette index of the entry pixel p maps to, from the item's label table
// (label_tables + the item's sorted-palette offset, one entry per sorted position).  The parameters after luts are only
// read by that instantiation.
template <bool kLabels>
__global__ void __launch_bounds__(kBatchThreads) batch_remap_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out,
                                                                     const BatchTile *tiles, const uint32_t *sorted, const uint2 *tables,
                                                                     const uint16_t *luts, const uint16_t *label_tables,
                                                                     uint32_t *__restrict__ labels) {
  __shared__ __align__(16) int4 s_ent[kIntColors];
  __shared__ int s_lut[kBatchLutEntries];
  __shared__ uint16_t s_lab[kLabels ? kIntColors : 1];
  const BatchTile t = tiles[blockIdx.x];
  const uint2 tab = tables[t.table];  // (offset of the item's sorted palette, its size)
  const int k = (int)tab.y;
  stage_palette_int(sorted + tab.x, k, s_ent);
  const uint16_t *lut = luts + (size_t)t.table * kBatchLutEntries;
  for (int i = threadIdx.x; i < kBatchLutEntries; i += kBatchThreads) s_lut[i] = (int)lut[i];
  if constexpr (kLabels)
    for (int i = threadIdx.x; i < k; i += kBatchThreads) s_lab[i] = label_tables[tab.x + i];
  __syncthreads();
  uint32_t c[kRemapPix];
  int lo[kRemapPix], hi[kRemapPix];
#pragma unroll
  for (int q = 0; q < kRemapPix; ++q) {
    const uint32_t p = t.begin + threadIdx.x + (uint32_t)q * kBatchThreads;
    c[q] = p < t.end ? (in[p] & 0x00FFFFFFu) : 0u;
  }
  nearest_int<kRemapPix>(s_ent, k, c, lo, hi);
#pragma unroll
  for (int q = 0; q < kRemapPix; ++q) {
    const uint32_t p = t.begin + threadIdx.x + (uint32_t)q * kBatchThreads;
    if (p < t.end) {
      const int win = resolve_int_index(s_ent, c[q], s_lut[((c[q] >> 16) & 0xFF) + ((c[q] >> 8) & 0xFF) + (c[q] & 0xFF)], lo[q], hi[q]);
      out[p] = (uint32_t)s_ent[win].w;
      if constexpr (kLabels) labels[p] = s_lab[win];
    }
  }
}

}  // namespace

void batch_hist_launch(const uint32_t *d_in, const BatchItem *d_items, uint32_t num_items, uint32_t *d_colours, uint32_t *d_counts,
                       uint32_t *d_first, uint32_t *d_res, cudaStream_t st) {
  DQ_RAISE_SMEM(batch_hist_kernel, kHistSmemBytes);
  batch_hist_kernel<<<num_items, kBatchThreads, kHistSmemBytes, st>>>(d_in, d_items, d_colours, d_counts, d_first, d_res);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void batch_split_launch(const BatchItem *d_items, uint32_t num_items, uint32_t max_points, const uint32_t *d_colours, uint32_t *d_counts,
                        const uint32_t *d_first, uint32_t *d_res, uint32_t *d_palette, uint32_t *d_cluster_size, double *d_cluster_mean,
                        cudaStream_t st) {
  const size_t smem = sizeof(exact::Shared);
  DQ_RAISE_SMEM(batch_split_kernel, smem);
  batch_split_kernel<<<num_items, kBatchThreads, smem, st>>>(d_items, std::min<uint32_t>(max_points, kBatchMaxPoints), d_colours, d_counts,
                                                            d_first, d_res, d_palette, d_cluster_size, d_cluster_mean);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void batch_remap_launch(const uint32_t *d_in, uint32_t *d_out, const BatchTile *d_tiles, uint32_t num_tiles, const uint32_t *d_sorted,
                        const uint2 *d_tables, const uint16_t *d_luts, const uint16_t *d_label_tables, uint32_t *d_labels,
                        cudaStream_t st) {
  if (d_labels != nullptr)
    batch_remap_kernel<true><<<num_tiles, kBatchThreads, 0, st>>>(d_in, d_out, d_tiles, d_sorted, d_tables, d_luts, d_label_tables,
                                                                  d_labels);
  else
    batch_remap_kernel<false><<<num_tiles, kBatchThreads, 0, st>>>(d_in, d_out, d_tiles, d_sorted, d_tables, d_luts, nullptr, nullptr);
  DQ_CUDA_CHECK(cudaGetLastError());
}

}  // namespace dq

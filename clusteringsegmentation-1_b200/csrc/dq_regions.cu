// dq_regions.cu -- stable partition of a tag image by region for dq_quant_regions_* and dq_map_regions_*: the pixel
// indexes sorted by tag, the pixels gathered in that order and the region offsets; afterwards the scatter of the
// quantized or mapped pixels and labels back.
//
// LSD radix sort of (tag, index) pairs, one pass per byte of the largest tag: 1 pass up to 256 regions, 2 up to 65 536,
// 3 up to 2^24.  A pass is the stable counting sort of dq_srm.cu over tiles of 2048 consecutive pairs:
//   count    per-tile histogram of the pass's digit          -> counts[digit][tile]
//   rowscan  exclusive scan of every digit's row + row total  (tile_rowscan_launch, shared with dq_srm.cu)
//   scatter  rank of a pair = digits before it + same-digit pairs of earlier tiles + same-digit pairs before it in its
//            tile (warp match -> per-segment counts -> per-digit running prefix over the tile's 64 segments)
// Every pass is stable, so region r's pixels come out in raster order: the order the single call and the batch see them
// in, on which the ordered split's first-seen ties depend.  The first pass reads the tags straight from the image and
// drops pixels whose tag is >= num_regions or whose region is set in the optional bitmap of dropped regions (the regions
// dq_map_regions does not map), so the later passes sort only the m pixels that lie in a kept region; they take m from
// the first pass's digit totals (the host does not know it until the offsets come back).  A dropped region comes out
// with no pixels.  The last pass also gathers in[index] into sorted order.
#include "dq_kernels.cuh"

namespace dq {
namespace {

constexpr int kThreads = kSortThreads;
constexpr int kSegs = 64;              // segments of 32 consecutive pairs per tile
constexpr int kTile = 32 * kSegs;      // 2048 pairs
constexpr int kSegsPerWarp = kSegs / (kThreads / 32);

struct RegionPass {
  const uint32_t *tags;     // first pass: the tag image
  const uint2 *src;         // later passes: the previous pass's (tag, index) pairs
  const uint32_t *m_total;  // later passes: the first pass's 256 digit totals, whose sum is the number of pairs
  const uint32_t *dropped;  // first pass: nullptr, or bit r of word r / 32 set = region r's pixels are dropped
  uint32_t n, num_regions, shift;
};

// Number of pairs the pass sorts (every thread of the CTA calls it; ends in a barrier).
template <bool kFirst>
__device__ __forceinline__ uint32_t pass_count(const RegionPass &p, uint32_t *warp_sum) {
  if (kFirst) return p.n;
  const uint32_t v = __reduce_add_sync(0xffffffffu, p.m_total[threadIdx.x]);
  if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = v;
  __syncthreads();
  uint32_t m = 0;
#pragma unroll
  for (int q = 0; q < kThreads / 32; ++q) m += warp_sum[q];
  __syncthreads();
  return m;
}

template <bool kFirst>
__device__ __forceinline__ bool load_pair(const RegionPass &p, uint32_t e, uint32_t m, uint32_t &tag, uint32_t &idx) {
  if (kFirst) {
    if (e >= p.n) return false;
    tag = p.tags[e];
    idx = e;
    return tag < p.num_regions && (p.dropped == nullptr || ((p.dropped[tag >> 5] >> (tag & 31u)) & 1u) == 0u);
  }
  if (e >= m) return false;
  const uint2 v = p.src[e];
  tag = v.x;
  idx = v.y;
  return true;
}

template <bool kFirst>
__global__ void __launch_bounds__(kThreads) region_count_kernel(const RegionPass p, uint32_t num_tiles, uint32_t *counts) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t warp_sum[kThreads / 32];
  hist[threadIdx.x] = 0;
  const uint32_t m = pass_count<kFirst>(p, warp_sum);
  __syncthreads();
  const uint32_t tile0 = blockIdx.x * kTile;
  for (uint32_t e = threadIdx.x; e < kTile; e += kThreads) {
    uint32_t tag = 0, idx = 0;
    if (load_pair<kFirst>(p, tile0 + e, m, tag, idx)) atomicAdd(&hist[(tag >> p.shift) & 0xFFu], 1u);
  }
  __syncthreads();
  counts[(size_t)threadIdx.x * num_tiles + blockIdx.x] = hist[threadIdx.x];
}

template <bool kFirst, bool kLast>
__global__ void __launch_bounds__(kThreads) region_scatter_kernel(const RegionPass p, uint32_t num_tiles,
                                                                  const uint32_t *__restrict__ counts,
                                                                  const uint32_t *__restrict__ row_total, uint2 *dst,
                                                                  const uint32_t *__restrict__ in, uint32_t *gathered) {
  __shared__ uint16_t seg[kSegs][256];  // per segment and digit: count, then exclusive prefix over the tile's segments
  __shared__ uint32_t bin_base[256];
  __shared__ uint32_t warp_sum[kThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < kSegs * 256 / 2; i += kThreads) reinterpret_cast<uint32_t *>(&seg[0][0])[i] = 0u;
  const uint32_t m = pass_count<kFirst>(p, warp_sum);
  // digits before mine: exclusive scan of the 256 row totals (thread = digit)
  {
    const uint32_t v = row_total[tid];
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    uint32_t before = 0;
    for (int q = 0; q < warp; ++q) before += warp_sum[q];
    bin_base[tid] = before + incl - v + counts[(size_t)tid * num_tiles + blockIdx.x];
  }
  __syncthreads();
  const uint32_t tile0 = blockIdx.x * kTile;
  uint32_t tag[kSegsPerWarp], idx[kSegsPerWarp], key[kSegsPerWarp];  // key = digit | rank_in_segment << 8 | valid << 16
#pragma unroll
  for (int k = 0; k < kSegsPerWarp; ++k) {
    const int sg = warp * kSegsPerWarp + k;
    tag[k] = idx[k] = 0;
    const bool valid = load_pair<kFirst>(p, tile0 + (uint32_t)sg * 32u + (uint32_t)lane, m, tag[k], idx[k]);
    const uint32_t d = valid ? (tag[k] >> p.shift) & 0xFFu : 256u;  // invalid lanes match only each other
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
    if (valid && rank == 0) seg[sg][d] = (uint16_t)__popc(peers);
    key[k] = d | (rank << 8) | ((uint32_t)valid << 16);
  }
  __syncthreads();
  {
    uint32_t running = 0;  // thread = digit: exclusive prefix over the segments, in order
#pragma unroll 8
    for (int sg = 0; sg < kSegs; ++sg) {
      const uint32_t c = seg[sg][tid];
      seg[sg][tid] = (uint16_t)running;
      running += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < kSegsPerWarp; ++k) {
    if (key[k] >> 16) {
      const int sg = warp * kSegsPerWarp + k;
      const uint32_t d = key[k] & 0xFFu, rank = (key[k] >> 8) & 0xFFu;
      const uint32_t at = bin_base[d] + seg[sg][d] + rank;
      dst[at] = make_uint2(tag[k], idx[k]);
      if (kLast) gathered[at] = in[idx[k]];
    }
  }
}

// offsets[r] = first sorted position of region r, offsets[num_regions] = m: the exclusive scan of the region sizes.  The
// thread at a change of tag writes the offsets of every region from the previous tag + 1 to its own (empty ones included).
__global__ void __launch_bounds__(kThreads) region_offsets_kernel(const uint2 *__restrict__ sorted, const uint32_t *__restrict__ m_total,
                                                                   uint32_t num_regions, uint32_t *offsets) {
  __shared__ uint32_t warp_sum[kThreads / 32];
  RegionPass p = {};
  p.m_total = m_total;
  const uint32_t m = pass_count<false>(p, warp_sum);
  for (uint32_t j = blockIdx.x * kThreads + threadIdx.x; j <= m; j += gridDim.x * kThreads) {
    const uint32_t lo = j == 0 ? 0u : sorted[j - 1].x + 1u;
    const uint32_t hi = j == m ? num_regions : sorted[j].x;
    for (uint32_t r = lo; r <= hi; ++r) offsets[r] = j;
  }
}

__global__ void __launch_bounds__(kThreads) region_scatter_back_kernel(const uint2 *__restrict__ sorted, uint32_t m,
                                                                        const uint32_t *__restrict__ g_out,
                                                                        const uint32_t *__restrict__ g_labels, uint32_t *out,
                                                                        uint32_t *labels) {
  const uint32_t j = blockIdx.x * kThreads + threadIdx.x;
  if (j >= m) return;
  const uint32_t p = sorted[j].y;
  out[p] = g_out[j];
  if (labels != nullptr) labels[p] = g_labels[j];
}

uint32_t region_tiles(uint32_t n) { return (uint32_t)(((size_t)n + kTile - 1) / kTile); }

}  // namespace

uint32_t region_passes(uint32_t num_regions) { return num_regions <= 256u ? 1u : num_regions <= 65536u ? 2u : 3u; }

size_t region_scratch_words(uint32_t n, uint32_t num_regions) {
  return (size_t)256 * region_tiles(n) + 512 + (size_t)num_regions + 1;
}

int region_partition(const uint32_t *d_in, const uint32_t *d_tags, uint32_t n, uint32_t num_regions, const uint32_t *d_dropped,
                     uint2 *d_pairs, uint32_t *d_gathered, uint32_t *d_scratch, const uint2 **d_sorted, cudaStream_t st) {
  const uint32_t tiles = region_tiles(n), passes = region_passes(num_regions);
  uint32_t *const counts = d_scratch, *const total0 = counts + (size_t)256 * tiles, *const total1 = total0 + 256;
  uint32_t *const offsets = total1 + 256;
  RegionPass p = {d_tags, nullptr, total0, d_dropped, n, num_regions, 0u};
  uint2 *dst = d_pairs;
  for (uint32_t pass = 0; pass < passes; ++pass) {
    const bool first = pass == 0, last = pass + 1 == passes;
    uint32_t *const row_total = first ? total0 : total1;
    dst = d_pairs + (size_t)(pass & 1u) * n;
    p.shift = 8u * pass;
    if (first) region_count_kernel<true><<<tiles, kThreads, 0, st>>>(p, tiles, counts);
    else region_count_kernel<false><<<tiles, kThreads, 0, st>>>(p, tiles, counts);
    tile_rowscan_launch(256, tiles, counts, row_total, st);
    if (first && last) region_scatter_kernel<true, true><<<tiles, kThreads, 0, st>>>(p, tiles, counts, row_total, dst, d_in, d_gathered);
    else if (first) region_scatter_kernel<true, false><<<tiles, kThreads, 0, st>>>(p, tiles, counts, row_total, dst, d_in, d_gathered);
    else if (last) region_scatter_kernel<false, true><<<tiles, kThreads, 0, st>>>(p, tiles, counts, row_total, dst, d_in, d_gathered);
    else region_scatter_kernel<false, false><<<tiles, kThreads, 0, st>>>(p, tiles, counts, row_total, dst, d_in, d_gathered);
    p.src = dst;
  }
  region_offsets_kernel<<<(uint32_t)(((size_t)n + kThreads) / kThreads), kThreads, 0, st>>>(dst, total0, num_regions, offsets);
  DQ_CUDA_CHECK(cudaGetLastError());
  *d_sorted = dst;
  return (int)(3 * passes + 1);
}

const uint32_t *region_offsets(const uint32_t *d_scratch, uint32_t n) { return d_scratch + (size_t)256 * region_tiles(n) + 512; }

void region_scatter_back(const uint2 *d_sorted, uint32_t m, const uint32_t *d_g_out, const uint32_t *d_g_labels, uint32_t *d_out,
                         uint32_t *d_labels, cudaStream_t st) {
  region_scatter_back_kernel<<<(m + kThreads - 1) / kThreads, kThreads, 0, st>>>(d_sorted, m, d_g_out, d_g_labels, d_out, d_labels);
  DQ_CUDA_CHECK(cudaGetLastError());
}

}  // namespace dq

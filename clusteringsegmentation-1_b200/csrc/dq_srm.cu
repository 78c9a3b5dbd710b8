// dq_srm.cu -- data-parallel front half of the reference's SRM (SURVEY.md 8f row 4): the edge list and its
// 256-bin counting sort.  The union-find merge loop that consumes the sorted edges stays on the host.
//
// Reference: SRM/srm.c
//   :103-121  diff(a, b) = max over the three colour bytes of |a - b|  (bytes at row*widthStep + channels*col)
//   :135-177  edge list: for every pixel of the (h-1) x (w-1) interior its right, then its lower neighbour; then the
//             last column's lower neighbours; then the last row's right neighbours
//   :226-246  bucket_sort: STABLE counting sort by diff -- the merge order, so the order inside a bucket is observable
//
// Three kernels over tiles of 2048 consecutive edges:
//   count    per-tile histogram of diff                      -> counts[bin][tile]
//   rowscan  exclusive scan of every bin's row + row total   (one CTA per bin; tile_rowscan_launch, also dq_regions.cu's)
//   scatter  rank of an edge = bins before it + same-bin edges of earlier tiles + same-bin edges before it in its
//            tile (warp match -> per-segment counts -> per-bin running prefix over the tile's 64 segments)
// 12 bytes written per edge, 2 x 3..4 bytes read per edge and pass (neighbouring reads hit L1/L2).
#include "dq_kernels.cuh"

namespace dq {
namespace {

constexpr int kSrmThreads = kSortThreads;
constexpr int kSrmSegs = 64;                 // segments of 32 consecutive edges per tile
constexpr int kSrmTile = 32 * kSrmSegs;      // 2048 edges
constexpr int kSrmSegsPerWarp = kSrmSegs / (kSrmThreads / 32);

struct SrmShape {
  uint32_t width, height, channels, width_step, interior, n_pairs;
};

__device__ __forceinline__ void edge_of(const SrmShape &s, uint32_t p, uint32_t &r1, uint32_t &r2) {
  if (p < s.interior) {
    const uint32_t q = p >> 1, i = q / (s.width - 1), j = q % (s.width - 1);
    r1 = i * s.width + j;
    r2 = (p & 1u) ? r1 + s.width : r1 + 1;
  } else if (p < s.interior + (s.height - 1)) {
    r1 = (p - s.interior) * s.width + s.width - 1;
    r2 = r1 + s.width;
  } else {
    r1 = (s.height - 1) * s.width + (p - s.interior - (s.height - 1));
    r2 = r1 + 1;
  }
}

__device__ __forceinline__ uint32_t edge_diff(const SrmShape &s, const uint8_t *__restrict__ in, uint32_t r1, uint32_t r2) {
  const uint8_t *a = in + (size_t)(r1 / s.width) * s.width_step + (size_t)s.channels * (r1 % s.width);
  const uint8_t *b = in + (size_t)(r2 / s.width) * s.width_step + (size_t)s.channels * (r2 % s.width);
  uint32_t d = 0;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int x = a[c], y = b[c];
    d = max(d, (uint32_t)abs(x - y));
  }
  return d;
}

__global__ void __launch_bounds__(kSrmThreads) srm_count_kernel(const SrmShape s, const uint8_t *__restrict__ in,
                                                                 uint32_t num_tiles, uint32_t *counts) {
  __shared__ uint32_t hist[256];
  hist[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t tile0 = blockIdx.x * kSrmTile;
  for (uint32_t e = threadIdx.x; e < kSrmTile; e += kSrmThreads) {
    const uint32_t p = tile0 + e;
    if (p < s.n_pairs) {
      uint32_t r1, r2;
      edge_of(s, p, r1, r2);
      atomicAdd(&hist[edge_diff(s, in, r1, r2)], 1u);
    }
  }
  __syncthreads();
  counts[(size_t)threadIdx.x * num_tiles + blockIdx.x] = hist[threadIdx.x];
}

// one CTA per bin: exclusive scan of counts[bin][0..num_tiles) in place, total to row_total[bin]
__global__ void __launch_bounds__(kSrmThreads) tile_rowscan_kernel(uint32_t num_tiles, uint32_t *counts, uint32_t *row_total) {
  __shared__ uint32_t warp_sum[kSrmThreads / 32];
  __shared__ uint32_t carry;
  uint32_t *row = counts + (size_t)blockIdx.x * num_tiles;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < num_tiles; base += kSrmThreads) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i < num_tiles ? row[i] : 0u;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    uint32_t before = carry;
    for (int q = 0; q < warp; ++q) before += warp_sum[q];
    if (i < num_tiles) row[i] = before + incl - v;
    __syncthreads();
    if (threadIdx.x == kSrmThreads - 1) carry = before + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) row_total[blockIdx.x] = carry;
}

__global__ void __launch_bounds__(kSrmThreads) srm_scatter_kernel(const SrmShape s, const uint8_t *__restrict__ in,
                                                                   uint32_t num_tiles, const uint32_t *__restrict__ counts,
                                                                   const uint32_t *__restrict__ row_total, uint32_t *out) {
  __shared__ uint16_t seg[kSrmSegs][256];  // per segment and bin: count, then exclusive prefix over the tile's segments
  __shared__ uint32_t bin_base[256];
  __shared__ uint32_t warp_sum[kSrmThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < kSrmSegs * 256 / 2; i += kSrmThreads) reinterpret_cast<uint32_t *>(&seg[0][0])[i] = 0u;
  // bins before mine: exclusive scan of the 256 row totals (thread = bin)
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
  const uint32_t tile0 = blockIdx.x * kSrmTile;
  uint32_t r1[kSrmSegsPerWarp], r2[kSrmSegsPerWarp], key[kSrmSegsPerWarp];  // key = diff | rank_in_segment << 8 | valid << 16
#pragma unroll
  for (int k = 0; k < kSrmSegsPerWarp; ++k) {
    const int sg = warp * kSrmSegsPerWarp + k;
    const uint32_t p = tile0 + (uint32_t)sg * 32u + (uint32_t)lane;
    const bool valid = p < s.n_pairs;
    uint32_t d = 256u;  // invalid lanes match only each other
    r1[k] = r2[k] = 0;
    if (valid) {
      edge_of(s, p, r1[k], r2[k]);
      d = edge_diff(s, in, r1[k], r2[k]);
    }
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
    if (valid && rank == 0) seg[sg][d] = (uint16_t)__popc(peers);
    key[k] = d | (rank << 8) | ((uint32_t)valid << 16);
  }
  __syncthreads();
  {
    uint32_t running = 0;  // thread = bin: exclusive prefix over the segments, in order
#pragma unroll 8
    for (int sg = 0; sg < kSrmSegs; ++sg) {
      const uint32_t c = seg[sg][tid];
      seg[sg][tid] = (uint16_t)running;
      running += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < kSrmSegsPerWarp; ++k) {
    if (key[k] >> 16) {
      const int sg = warp * kSrmSegsPerWarp + k;
      const uint32_t d = key[k] & 0xFFu, rank = (key[k] >> 8) & 0xFFu;
      const size_t at = (size_t)bin_base[d] + seg[sg][d] + rank;
      out[3 * at] = r1[k];
      out[3 * at + 1] = r2[k];
      out[3 * at + 2] = d;
    }
  }
}

}  // namespace

void tile_rowscan_launch(uint32_t num_bins, uint32_t num_tiles, uint32_t *counts, uint32_t *row_total, cudaStream_t st) {
  tile_rowscan_kernel<<<num_bins, kSrmThreads, 0, st>>>(num_tiles, counts, row_total);
}

uint32_t srm_num_pairs(uint32_t width, uint32_t height) {
  return 2u * (width - 1u) * (height - 1u) + (height - 1u) + (width - 1u);  // srm.c:58
}

size_t srm_scratch_words(uint32_t width, uint32_t height) {
  const uint32_t n = srm_num_pairs(width, height);
  const size_t tiles = ((size_t)n + kSrmTile - 1) / kSrmTile;
  return 256 * tiles + 256;
}

int srm_sorted_edges(const uint8_t *d_in, uint32_t width, uint32_t height, uint32_t channels, uint32_t width_step,
                     uint32_t *d_pairs, uint32_t *d_scratch, cudaStream_t st) {
  SrmShape s;
  s.width = width;
  s.height = height;
  s.channels = channels;
  s.width_step = width_step;
  s.interior = 2u * (width - 1u) * (height - 1u);
  s.n_pairs = srm_num_pairs(width, height);
  if (s.n_pairs == 0) return 0;
  const uint32_t tiles = (s.n_pairs + kSrmTile - 1) / kSrmTile;
  uint32_t *counts = d_scratch, *row_total = d_scratch + (size_t)256 * tiles;
  srm_count_kernel<<<tiles, kSrmThreads, 0, st>>>(s, d_in, tiles, counts);
  tile_rowscan_launch(256, tiles, counts, row_total, st);
  srm_scatter_kernel<<<tiles, kSrmThreads, 0, st>>>(s, d_in, tiles, counts, row_total, d_pairs);
  DQ_CUDA_CHECK(cudaGetLastError());
  return 3;
}

}  // namespace dq

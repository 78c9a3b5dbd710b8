// dq_map.cu -- nearest-palette remap.
//
// Reference: map_colors_mps, DivQuant/DivQuantMapColors.cpp:243-539.  The reference sorts the palette
// by r+g+b, starts at lut_init[r+g+b] and walks up/down alternately, pruning with (delta sum)^2/3.
// Its result is exactly  argmin_k (dist(k), rank(k))  over the WHOLE sorted palette, with
// rank(s)=0, rank(s+d)=2d-1, rank(s-d)=2d (SURVEY.md 8a; re-verified against the compiled reference
// in tests/test_oracle_golden.py), because the prune bound never exceeds the true distance and a
// candidate only replaces the incumbent when strictly closer.
//
// The sorted palette and lut_init come from the host shim, which calls the same std::sort as the
// reference (the order of equal sums is observable, SURVEY.md 7).
//
// Two device formulations, both bit-exact:
//   * brute force over pixels (map_pixels_*): N*K distance evaluations.
//   * de-duplicated (map_unique + map_gather): the K evaluations are done once per UNIQUE colour and
//     the answer is parked in the 2^24-entry direct table; pixels then gather through it.  Used
//     whenever a histogram of the same pixels is at hand (quant_recurse always has one).
#include <algorithm>
#include <atomic>

#include "dq_kernels.cuh"
#include "dq_map_int.cuh"

namespace dq {
namespace {

constexpr int kMapThreads = 256;
constexpr uint32_t kLutEntries = 3 * 255 + 1;

// Winner in the sorted palette for one colour.  `pal` holds {r, g, b, packed 0x00RRGGBB}.
__device__ __forceinline__ uint32_t nearest_entry(uint32_t colour, const int4 *pal, int num_colors, const int *lut) {
  const int r = (colour >> 16) & 0xFF, g = (colour >> 8) & 0xFF, b = colour & 0xFF;
  const int s = lut[r + g + b];
  // lexicographic (dist, rank): dist < 2^18, rank < 2K
  uint64_t best = ~uint64_t(0);
  int win = s;
#pragma unroll 4
  for (int k = 0; k < num_colors; ++k) {
    const int4 e = pal[k];
    const int dr = r - e.x, dg = g - e.y, db = b - e.z;
    const uint32_t dist = (uint32_t)(dr * dr + dg * dg + db * db);
    const uint32_t rank = (k > s) ? (uint32_t)(2 * (k - s) - 1) : (uint32_t)(2 * (s - k));
    const uint64_t key = ((uint64_t)dist << 32) | rank;
    if (key < best) {
      best = key;
      win = k;
    }
  }
  return (uint32_t)pal[win].w;
}

__device__ __forceinline__ void stage_palette(const uint32_t *sorted, int num_colors, const int *lut_init, int4 *s_pal,
                                              int *s_lut) {
  for (int k = threadIdx.x; k < num_colors; k += blockDim.x) {
    const uint32_t c = sorted[k] & 0x00FFFFFFu;
    s_pal[k] = make_int4((c >> 16) & 0xFF, (c >> 8) & 0xFF, c & 0xFF, (int)c);
  }
  for (int i = threadIdx.x; i < (int)kLutEntries; i += blockDim.x) s_lut[i] = lut_init[i];
  __syncthreads();
}

// ---- fast formulation (palette in shared memory) --------------------------------------------------
// dist(k) - |p|^2 = |c_k|^2 - 2 p.c_k is linear in the pixel, so with the palette pre-expanded to
// {-2r, -2g, -2b, r^2+g^2+b^2} one evaluation is 3 FFMA + 1 FMNMX (all values are integers below 2^24 in
// magnitude, hence exact in FP32) -- the "4 lane-instructions per evaluation" of SURVEY.md 8d.  One
// broadcast LDS.128 per palette entry is shared by PIX pixels of the thread.  The arg-min with the
// reference's tie-break is then found by walking the reference's own visiting order (start index, +1, -1,
// +2, ...) until the first entry at the minimal distance: that entry is argmin (dist, rank) by definition.
template <int PIX>
struct PixelBlock {
  float r[PIX], g[PIX], b[PIX], best[PIX];
};

__device__ __forceinline__ float entry_key(const float4 e, float r, float g, float b) {
  return fmaf(r, e.x, fmaf(g, e.y, fmaf(b, e.z, e.w)));
}

template <int PIX>
__device__ __forceinline__ void min_distance(const float4 *s_pal, int num_colors, PixelBlock<PIX> &px) {
#pragma unroll
  for (int i = 0; i < PIX; ++i) px.best[i] = 3.0e38f;
#pragma unroll 8
  for (int k = 0; k < num_colors; ++k) {
    const float4 e = s_pal[k];
#pragma unroll
    for (int i = 0; i < PIX; ++i) px.best[i] = fminf(px.best[i], entry_key(e, px.r[i], px.g[i], px.b[i]));
  }
}

// First entry, in the reference's visiting order from start index s, whose distance equals the minimum.
__device__ __forceinline__ int first_at_minimum(const float4 *s_pal, int num_colors, int s, float r, float g, float b,
                                                float best) {
  if (entry_key(s_pal[s], r, g, b) == best) return s;
  for (int d = 1; d < num_colors; ++d) {
    const int up = s + d, down = s - d;
    if (up < num_colors && entry_key(s_pal[up], r, g, b) == best) return up;
    if (down >= 0 && entry_key(s_pal[down], r, g, b) == best) return down;
  }
  return s;  // unreachable: the minimum is attained by some entry
}

template <typename LutT>
__device__ __forceinline__ void stage_palette_fast(const uint32_t *sorted, int num_colors, const LutT *lut_init,
                                                   float4 *s_pal, uint32_t *s_word, int *s_lut) {
  for (int k = threadIdx.x; k < num_colors; k += blockDim.x) {
    const uint32_t c = sorted[k] & 0x00FFFFFFu;
    const float r = (float)((c >> 16) & 0xFF), g = (float)((c >> 8) & 0xFF), b = (float)(c & 0xFF);
    s_pal[k] = make_float4(-2.f * r, -2.f * g, -2.f * b, r * r + g * g + b * b);
    s_word[k] = c;
  }
  for (int i = threadIdx.x; i < (int)kLutEntries; i += blockDim.x) s_lut[i] = (int)lut_init[i];
  __syncthreads();
}


constexpr int kFastPix = 8;  // pixels per thread per iteration: two 128-bit loads

__global__ void __launch_bounds__(kMapThreads) map_pixels_fast_kernel(const uint32_t *__restrict__ in, uint32_t n,
                                                                     uint32_t *__restrict__ out, const uint32_t *sorted,
                                                                     int num_colors, const int *lut_init) {
  extern __shared__ __align__(16) unsigned char smem[];
  float4 *s_pal = reinterpret_cast<float4 *>(smem);
  uint32_t *s_word = reinterpret_cast<uint32_t *>(smem + (size_t)num_colors * 16);
  int *s_lut = reinterpret_cast<int *>(smem + (size_t)num_colors * 20);
  const uint32_t nblk = n / kFastPix;
  const uint4 *in4 = reinterpret_cast<const uint4 *>(in);
  uint4 *out4 = reinterpret_cast<uint4 *>(out);
  if (num_colors <= kIntColors) {
    int4 *s_ent = reinterpret_cast<int4 *>(smem);
    s_lut = reinterpret_cast<int *>(smem + (size_t)((num_colors + 1) & ~1) * 16);
    stage_palette_int(sorted, num_colors, s_ent);
    for (int i = threadIdx.x; i < (int)kLutEntries; i += blockDim.x) s_lut[i] = lut_init[i];
    __syncthreads();
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < nblk; t += gridDim.x * blockDim.x) {
      const uint4 a = __ldcs(in4 + 2 * t), c = __ldcs(in4 + 2 * t + 1);
      const uint32_t w[kFastPix] = {a.x & 0xFFFFFFu, a.y & 0xFFFFFFu, a.z & 0xFFFFFFu, a.w & 0xFFFFFFu,
                                    c.x & 0xFFFFFFu, c.y & 0xFFFFFFu, c.z & 0xFFFFFFu, c.w & 0xFFFFFFu};
      int lo[kFastPix], hi[kFastPix];
      nearest_int<kFastPix>(s_ent, num_colors, w, lo, hi);
      uint32_t res[kFastPix];
#pragma unroll
      for (int i = 0; i < kFastPix; ++i)
        res[i] = resolve_int(s_ent, w[i], s_lut[((w[i] >> 16) & 0xFF) + ((w[i] >> 8) & 0xFF) + (w[i] & 0xFF)], lo[i], hi[i]);
      __stcs(out4 + 2 * t, make_uint4(res[0], res[1], res[2], res[3]));
      __stcs(out4 + 2 * t + 1, make_uint4(res[4], res[5], res[6], res[7]));
    }
    const uint32_t tail = nblk * kFastPix;
    if (blockIdx.x == 0 && tail + threadIdx.x < n) {
      const uint32_t w[1] = {in[tail + threadIdx.x] & 0xFFFFFFu};
      int lo[1], hi[1];
      nearest_int<1>(s_ent, num_colors, w, lo, hi);
      out[tail + threadIdx.x] = resolve_int(s_ent, w[0], s_lut[((w[0] >> 16) & 0xFF) + ((w[0] >> 8) & 0xFF) + (w[0] & 0xFF)], lo[0], hi[0]);
    }
    return;
  }
  stage_palette_fast(sorted, num_colors, lut_init, s_pal, s_word, s_lut);
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < nblk; t += gridDim.x * blockDim.x) {
    const uint4 a = __ldcs(in4 + 2 * t), c = __ldcs(in4 + 2 * t + 1);
    const uint32_t w[kFastPix] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
    PixelBlock<kFastPix> px;
    int start[kFastPix];
#pragma unroll
    for (int i = 0; i < kFastPix; ++i) {
      const int R = (w[i] >> 16) & 0xFF, G = (w[i] >> 8) & 0xFF, B = w[i] & 0xFF;
      px.r[i] = (float)R, px.g[i] = (float)G, px.b[i] = (float)B;
      start[i] = s_lut[R + G + B];
    }
    min_distance<kFastPix>(s_pal, num_colors, px);
    uint32_t res[kFastPix];
#pragma unroll
    for (int i = 0; i < kFastPix; ++i)
      res[i] = s_word[first_at_minimum(s_pal, num_colors, start[i], px.r[i], px.g[i], px.b[i], px.best[i])];
    __stcs(out4 + 2 * t, make_uint4(res[0], res[1], res[2], res[3]));
    __stcs(out4 + 2 * t + 1, make_uint4(res[4], res[5], res[6], res[7]));
  }
  // tail: fewer than kFastPix pixels, one thread each
  const uint32_t tail0 = nblk * kFastPix;
  if (blockIdx.x == 0 && tail0 + threadIdx.x < n) {
    const uint32_t wv = in[tail0 + threadIdx.x];
    const int R = (wv >> 16) & 0xFF, G = (wv >> 8) & 0xFF, B = wv & 0xFF;
    PixelBlock<1> px;
    px.r[0] = (float)R, px.g[0] = (float)G, px.b[0] = (float)B;
    min_distance<1>(s_pal, num_colors, px);
    out[tail0 + threadIdx.x] = s_word[first_at_minimum(s_pal, num_colors, s_lut[R + G + B], px.r[0], px.g[0], px.b[0], px.best[0])];
  }
}

constexpr int kUniqInt = 2;  // colours per thread of the integer formulation (4K K=256, 125 712 colours: 1 -> 25 us, 2 -> 22 us, 4 -> 29 us)
constexpr int kUniqPix = 2;  // colours per thread (measured at 4K, K=256: 4 -> 26 us, 2 -> 22 us, 1 -> 25 us)

// One evaluation per unique colour: body shared by the two ways the tables arrive.
template <typename LutT>
__device__ __forceinline__ void map_unique_fast_body(const uint32_t *__restrict__ uniq, const uint32_t *ucount, uint32_t *table,
                                                     const uint32_t *sorted, int num_colors, const LutT *lut_init) {
  extern __shared__ __align__(16) unsigned char smem[];
  float4 *s_pal = reinterpret_cast<float4 *>(smem);
  uint32_t *s_word = reinterpret_cast<uint32_t *>(smem + (size_t)num_colors * 16);
  int *s_lut = reinterpret_cast<int *>(smem + (size_t)num_colors * 20);
  const uint32_t u = *ucount;
  const uint32_t stride = gridDim.x * blockDim.x;
  if (num_colors <= kIntColors) {
    int4 *s_ent = reinterpret_cast<int4 *>(smem);
    s_lut = reinterpret_cast<int *>(smem + (size_t)((num_colors + 1) & ~1) * 16);
    stage_palette_int(sorted, num_colors, s_ent);
    for (int i = threadIdx.x; i < (int)kLutEntries; i += blockDim.x) s_lut[i] = (int)lut_init[i];
    __syncthreads();
    for (uint32_t base = blockIdx.x * blockDim.x + threadIdx.x; base < u; base += kUniqInt * stride) {
      uint32_t c[kUniqInt];
      int lo[kUniqInt], hi[kUniqInt];
#pragma unroll
      for (int i = 0; i < kUniqInt; ++i) {
        const uint32_t idx = base + (uint32_t)i * stride;
        c[i] = idx < u ? (uniq[idx] & 0xFFFFFFu) : 0u;
      }
      nearest_int<kUniqInt>(s_ent, num_colors, c, lo, hi);
#pragma unroll
      for (int i = 0; i < kUniqInt; ++i) {
        if (base + (uint32_t)i * stride < u)
          table[c[i]] = 0x80000000u |
                        resolve_int(s_ent, c[i], s_lut[((c[i] >> 16) & 0xFF) + ((c[i] >> 8) & 0xFF) + (c[i] & 0xFF)], lo[i], hi[i]);
      }
    }
    return;
  }
  stage_palette_fast(sorted, num_colors, lut_init, s_pal, s_word, s_lut);
  // every thread takes kUniqPix colours a stride apart (coalesced loads of the unique list)
  for (uint32_t base = blockIdx.x * blockDim.x + threadIdx.x; base < u; base += kUniqPix * stride) {
    uint32_t c[kUniqPix];
    PixelBlock<kUniqPix> px;
    int start[kUniqPix];
#pragma unroll
    for (int i = 0; i < kUniqPix; ++i) {
      const uint32_t idx = base + (uint32_t)i * stride;
      c[i] = idx < u ? uniq[idx] : 0u;
      const int R = (c[i] >> 16) & 0xFF, G = (c[i] >> 8) & 0xFF, B = c[i] & 0xFF;
      px.r[i] = (float)R, px.g[i] = (float)G, px.b[i] = (float)B;
      start[i] = s_lut[R + G + B];
    }
    min_distance<kUniqPix>(s_pal, num_colors, px);
#pragma unroll
    for (int i = 0; i < kUniqPix; ++i) {
      if (base + (uint32_t)i * stride < u)
        table[c[i]] = 0x80000000u | s_word[first_at_minimum(s_pal, num_colors, start[i], px.r[i], px.g[i], px.b[i], px.best[i])];
    }
  }
}

__global__ void __launch_bounds__(kMapThreads) map_unique_fast_kernel(const uint32_t *__restrict__ uniq, const uint32_t *ucount,
                                                                     uint32_t *table, const uint32_t *sorted, int num_colors,
                                                                     const int *lut_init) {
  map_unique_fast_body(uniq, ucount, table, sorted, num_colors, lut_init);
}

// Tables inside the parameter block (constant bank): K <= 256.
__global__ void __launch_bounds__(kMapThreads) map_unique_fast_param_kernel(const __grid_constant__ MapTablesParam tables,
                                                                           const uint32_t *__restrict__ uniq,
                                                                           const uint32_t *ucount, uint32_t *table,
                                                                           int num_colors) {
  map_unique_fast_body(uniq, ucount, table, tables.sorted, num_colors, tables.lut);
}

inline size_t fast_smem_bytes(int num_colors) { return (size_t)num_colors * 20 + kLutEntries * 4 + 64; }  // covers both layouts

// Brute force over pixels, palette staged in shared memory.
__global__ void __launch_bounds__(kMapThreads) map_pixels_kernel(const uint32_t *__restrict__ in, uint32_t n,
                                                                uint32_t *__restrict__ out, const uint32_t *sorted,
                                                                int num_colors, const int *lut_init) {
  extern __shared__ __align__(16) unsigned char smem[];
  int *s_lut = reinterpret_cast<int *>(smem);
  int4 *s_pal = reinterpret_cast<int4 *>(smem + ((kLutEntries * 4 + 15) & ~15u));
  stage_palette(sorted, num_colors, lut_init, s_pal, s_lut);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    out[i] = nearest_entry(in[i], s_pal, num_colors, s_lut);
}

// Same, palette read from global memory (palettes too large for shared memory).
__global__ void __launch_bounds__(kMapThreads) map_pixels_big_kernel(const uint32_t *__restrict__ in, uint32_t n,
                                                                    uint32_t *__restrict__ out, const int4 *pal,
                                                                    int num_colors, const int *lut_init) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    out[i] = nearest_entry(in[i], pal, num_colors, lut_init);
}

// One evaluation per unique colour, palette read from global memory (palettes too large for shared memory).
__global__ void __launch_bounds__(kMapThreads) map_unique_big_kernel(const uint32_t *__restrict__ uniq, const uint32_t *ucount,
                                                                    uint32_t *table, const int4 *pal, int num_colors,
                                                                    const int *lut_init) {
  const uint32_t u = *ucount;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < u; i += gridDim.x * blockDim.x) {
    const uint32_t c = uniq[i] & 0xFFFFFFu;
    table[c] = 0x80000000u | nearest_entry(c, pal, num_colors, lut_init);
  }
}

__global__ void __launch_bounds__(kMapThreads) expand_palette_kernel(const uint32_t *sorted, int num_colors, int4 *pal) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < num_colors; k += gridDim.x * blockDim.x) {
    const uint32_t c = sorted[k] & 0x00FFFFFFu;
    pal[k] = make_int4((c >> 16) & 0xFF, (c >> 8) & 0xFF, c & 0xFF, (int)c);
  }
}

__global__ void __launch_bounds__(kMapThreads) map_gather_kernel(const uint32_t *__restrict__ in, uint32_t n,
                                                                uint32_t *__restrict__ out, const uint32_t *table,
                                                                uint32_t word_mask, uint32_t shift) {
  // 4 pixels per thread: one streaming 128-bit load, four table reads (the table entries of an image's colours
  // live in L2), one streaming 128-bit store.  (8 per thread measured slower: 35 vs 28 us at 4K.)
  const uint32_t nvec = n >> 2;
  const uint4 *in4 = reinterpret_cast<const uint4 *>(in);
  uint4 *out4 = reinterpret_cast<uint4 *>(out);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += gridDim.x * blockDim.x) {
    const uint4 p = __ldcs(in4 + i);
    uint4 q;
    q.x = table[(p.x & word_mask) >> shift] & 0x00FFFFFFu;
    q.y = table[(p.y & word_mask) >> shift] & 0x00FFFFFFu;
    q.z = table[(p.z & word_mask) >> shift] & 0x00FFFFFFu;
    q.w = table[(p.w & word_mask) >> shift] & 0x00FFFFFFu;
    __stcs(out4 + i, q);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3u)) {
    const uint32_t i = (nvec << 2) + threadIdx.x;
    out[i] = table[(in[i] & word_mask) >> shift] & 0x00FFFFFFu;
  }
}

__global__ void __launch_bounds__(kMapThreads) map_gather_scalar_kernel(const uint32_t *__restrict__ in, uint32_t n,
                                                                       uint32_t *__restrict__ out, const uint32_t *table) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    out[i] = table[in[i] & 0x00FFFFFFu] & 0x00FFFFFFu;
}

// ---- block majority vote (genHistogramsForBlocks, ClusteringSegmentation.cpp:417-563) ------------------------
// One thread per block.  The reference counts in a std::unordered_map<uint32_t,uint32_t> and takes the first
// maximum in ITERATION order, so that order is reproduced: libstdc++ keeps one singly linked list; a new key
// whose bucket (key % bucket_count, identity hash) is empty goes to the front of the whole list, otherwise to the
// front of its bucket's run; the table starts with 1 bucket, grows to the next prime >= max(n+1, 2*buckets) when
// n+1 would exceed the bucket count, and a rehash re-inserts the nodes in list order by the same rule.
constexpr int kVoteMaxKeys = 64;  // superpixelDim <= 8

__device__ __forceinline__ uint32_t next_bucket_count(uint32_t want) {
  // the entries of libstdc++'s prime table that matter below 2*64
  const uint32_t primes[] = {2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37, 41, 43, 47, 53, 59, 61, 67, 71, 73, 79, 83, 89, 97, 103, 109, 113, 127, 137, 139, 149, 157, 167};
  for (uint32_t p : primes) if (p >= want) return p;
  return 167;
}

__device__ __forceinline__ void list_insert(const uint32_t *keys, int *ord, int n_in_list, int e, uint32_t nb) {
  const uint32_t b = keys[e] % nb;
  int pos = 0;  // empty bucket: front of the list
  for (int i = 0; i < n_in_list; ++i) {
    if (keys[ord[i]] % nb == b) {
      pos = i;  // front of that bucket's run
      break;
    }
  }
  for (int i = n_in_list; i > pos; --i) ord[i] = ord[i - 1];
  ord[pos] = e;
}

__global__ void __launch_bounds__(128) block_vote_kernel(const uint32_t *__restrict__ quant, uint32_t width, uint32_t height,
                                                        uint32_t dim, uint32_t bw, uint32_t bh, uint32_t *__restrict__ blocks) {
  const uint32_t blk = blockIdx.x * blockDim.x + threadIdx.x;
  if (blk >= bw * bh) return;
  const uint32_t bx = blk % bw, by = blk / bw;
  uint32_t keys[kVoteMaxKeys], counts[kVoteMaxKeys];
  int ord[kVoteMaxKeys], tmp[kVoteMaxKeys];
  int n = 0;
  uint32_t nb = 1, resize_at = 0;  // default-constructed table: 1 bucket, first insert rehashes
  for (uint32_t y = by * dim; y < by * dim + dim && y < height; ++y) {
    for (uint32_t x = bx * dim; x < bx * dim + dim && x < width; ++x) {
      const uint32_t q = quant[(size_t)y * width + x];
      int found = -1;
      for (int i = 0; i < n; ++i) if (keys[i] == q) found = i;
      if (found >= 0) {
        counts[found] += 1;
        continue;
      }
      if ((uint32_t)n + 1 > resize_at) {
        nb = next_bucket_count(max((uint32_t)n + 1, nb * 2));
        if (n == 0) nb = 13;  // _Prime_rehash_policy: the first insertion always lands on 13 buckets
        resize_at = nb;       // max_load_factor 1.0
        for (int i = 0; i < n; ++i) tmp[i] = ord[i];
        for (int i = 0; i < n; ++i) list_insert(keys, ord, i, tmp[i], nb);
      }
      keys[n] = q;
      counts[n] = 1;
      list_insert(keys, ord, n, n, nb);
      ++n;
    }
  }
  // all-same blocks fall out naturally (one key); otherwise the first strict maximum in iteration order (:535-547)
  uint32_t best = 0;
  int max_count = 0;
  for (int i = 0; i < n; ++i) {
    const int e = ord[i];
    if ((int)counts[e] > max_count) {
      max_count = (int)counts[e];
      best = keys[e];
    }
  }
  blocks[blk] = best;
}

// Label image: binary search of every pixel in the palette sorted by colour value ((colour, last index) pairs).
__global__ void __launch_bounds__(kMapThreads) map_labels_kernel(const uint32_t *__restrict__ in, uint32_t n,
                                                                uint32_t *__restrict__ out, const uint2 *pairs, int num_pairs,
                                                                int greyscale, uint32_t *error) {
  extern __shared__ __align__(16) unsigned char smem[];
  uint2 *s_pairs = reinterpret_cast<uint2 *>(smem);
  for (int i = threadIdx.x; i < num_pairs; i += blockDim.x) s_pairs[i] = pairs[i];
  __syncthreads();
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t c = in[i] & 0x00FFFFFFu;
    int lo = 0, hi = num_pairs - 1, found = -1;
    while (lo <= hi) {
      const int mid = (lo + hi) >> 1;
      const uint32_t v = s_pairs[mid].x;
      if (v == c) {
        found = (int)s_pairs[mid].y;
        break;
      }
      if (v < c) lo = mid + 1; else hi = mid - 1;
    }
    if (found < 0) {
      atomicMax(error, i + 1u);
      found = 0;
    }
    out[i] = greyscale ? ((uint32_t)found << 16) | ((uint32_t)found << 8) | (uint32_t)found : (uint32_t)found;
  }
}

inline int blocks_for(uint64_t items, int threads, int sm_count, int per_sm) {
  uint64_t want = (items + threads - 1) / threads;
  uint64_t cap = (uint64_t)sm_count * per_sm;
  if (want < 1) want = 1;
  return (int)(want < cap ? want : cap);
}

inline size_t map_smem_bytes(int num_colors) { return ((kLutEntries * 4 + 15) & ~15u) + (size_t)num_colors * sizeof(int4); }

}  // namespace

int map_smem_palette_limit() { return 8192; }  // 160 KB of expanded entries + the LUT fit the 227 KB carve-out

void map_pixels(const uint32_t *d_in, uint32_t n, uint32_t *d_out, const uint32_t *d_sorted, int num_colors,
                const int *d_lut, int4 *d_pal_scratch, int sm_count, cudaStream_t st) {
  if (n == 0) return;
  const bool aligned = ((reinterpret_cast<uintptr_t>(d_in) | reinterpret_cast<uintptr_t>(d_out)) & 15u) == 0;
  if (num_colors <= map_smem_palette_limit() && aligned) {
    const size_t smem = fast_smem_bytes(num_colors);
    DQ_RAISE_SMEM(map_pixels_fast_kernel, smem);
    // resident CTAs per SM are bounded by the palette's shared memory; keep the grid a multiple of the SM count
    int per_sm = (int)std::min<size_t>(8, std::max<size_t>(1, (200 * 1024) / smem));
    map_pixels_fast_kernel<<<blocks_for(n / kFastPix + 1, kMapThreads, sm_count, per_sm), kMapThreads, smem, st>>>(
        d_in, n, d_out, d_sorted, num_colors, d_lut);
  } else if (num_colors <= map_smem_palette_limit()) {
    const size_t smem = map_smem_bytes(num_colors);
    DQ_RAISE_SMEM(map_pixels_kernel, smem);
    map_pixels_kernel<<<blocks_for(n, kMapThreads, sm_count, 8), kMapThreads, smem, st>>>(d_in, n, d_out, d_sorted,
                                                                                         num_colors, d_lut);
  } else {
    expand_palette_kernel<<<blocks_for(num_colors, kMapThreads, sm_count, 1), kMapThreads, 0, st>>>(d_sorted, num_colors,
                                                                                                   d_pal_scratch);
    map_pixels_big_kernel<<<blocks_for(n, kMapThreads, sm_count, 8), kMapThreads, 0, st>>>(d_in, n, d_out, d_pal_scratch,
                                                                                          num_colors, d_lut);
  }
  DQ_CUDA_CHECK(cudaGetLastError());
}

void map_unique(const uint32_t *d_uniq, const uint32_t *d_ucount, uint32_t u_hint, uint32_t *d_table,
                const uint32_t *d_sorted, int num_colors, const int *d_lut, int4 *d_pal_scratch, int sm_count, cudaStream_t st) {
  if (num_colors > map_smem_palette_limit()) {
    expand_palette_kernel<<<blocks_for(num_colors, kMapThreads, sm_count, 1), kMapThreads, 0, st>>>(d_sorted, num_colors,
                                                                                                   d_pal_scratch);
    map_unique_big_kernel<<<blocks_for(u_hint, kMapThreads, sm_count, 8), kMapThreads, 0, st>>>(d_uniq, d_ucount, d_table,
                                                                                               d_pal_scratch, num_colors, d_lut);
    DQ_CUDA_CHECK(cudaGetLastError());
    return;
  }
  const size_t smem = fast_smem_bytes(num_colors);
  DQ_RAISE_SMEM(map_unique_fast_kernel, smem);
  int per_sm = (int)std::min<size_t>(8, std::max<size_t>(1, (200 * 1024) / smem));
  map_unique_fast_kernel<<<blocks_for(u_hint / kUniqPix + 1, kMapThreads, sm_count, per_sm), kMapThreads, smem, st>>>(
      d_uniq, d_ucount, d_table, d_sorted, num_colors, d_lut);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void map_unique_params(const MapTablesParam &tables, const uint32_t *d_uniq, const uint32_t *d_ucount, uint32_t u_hint,
                       uint32_t *d_table, int num_colors, int sm_count, cudaStream_t st) {
  const size_t smem = fast_smem_bytes(num_colors);  // <= 256 colours: below 48 KB
  int per_sm = (int)std::min<size_t>(8, std::max<size_t>(1, (200 * 1024) / smem));
  map_unique_fast_param_kernel<<<blocks_for(u_hint / kUniqPix + 1, kMapThreads, sm_count, per_sm), kMapThreads, smem, st>>>(
      tables, d_uniq, d_ucount, d_table, num_colors);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void block_vote(const uint32_t *d_quant, uint32_t width, uint32_t height, uint32_t dim, uint32_t *d_blocks, int sm_count,
                cudaStream_t st) {
  const uint32_t bw = (width + dim - 1) / dim, bh = (height + dim - 1) / dim;
  (void)sm_count;
  block_vote_kernel<<<(bw * bh + 127) / 128, 128, 0, st>>>(d_quant, width, height, dim, bw, bh, d_blocks);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void map_labels(const uint32_t *d_in, uint32_t n, uint32_t *d_out, const uint2 *d_pairs, int num_pairs, int greyscale,
                uint32_t *d_error, int sm_count, cudaStream_t st) {
  if (n == 0) return;
  const size_t smem = (size_t)num_pairs * sizeof(uint2);
  DQ_RAISE_SMEM(map_labels_kernel, smem);
  map_labels_kernel<<<blocks_for(n, kMapThreads, sm_count, 4), kMapThreads, smem, st>>>(d_in, n, d_out, d_pairs, num_pairs,
                                                                                       greyscale, d_error);
  DQ_CUDA_CHECK(cudaGetLastError());
}

void map_gather(const uint32_t *d_in, uint32_t n, uint32_t *d_out, const uint32_t *d_table, int sm_count, cudaStream_t st) {
  if (n == 0) return;
  const bool aligned = ((reinterpret_cast<uintptr_t>(d_in) | reinterpret_cast<uintptr_t>(d_out)) & 15u) == 0;
  if (aligned)
    map_gather_kernel<<<blocks_for((n >> 2) + 1, kMapThreads, sm_count, 8), kMapThreads, 0, st>>>(d_in, n, d_out, d_table,
                                                                                                 0x00FFFFFFu, 0u);
  else
    map_gather_scalar_kernel<<<blocks_for(n, kMapThreads, sm_count, 8), kMapThreads, 0, st>>>(d_in, n, d_out, d_table);
  DQ_CUDA_CHECK(cudaGetLastError());
}

}  // namespace dq

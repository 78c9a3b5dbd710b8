// dq_map_int.cuh -- the keyed integer arg-min of the remap (palettes of at most 512 entries), shared by the remap kernels
// of dq_map.cu and the batch remap of dq_batch.cu.
#pragma once

#include "dq_common.cuh"

namespace dq {

// ---- integer formulation (K <= 512) -------------------------------------------------------------------------
// With the colour bytes packed in one word,  p.c_k  is ONE dp4a, and  2 p.c_k - |c_k|^2 = |p|^2 - dist(k)  grows as the
// distance shrinks.  The entry index rides in the low 9 bits of the key, so the arg-min needs no second pass:
//   key_lo = (2 p.c_k - |c_k|^2) * 512 + (511 - k) : the maximum names the SMALLEST k at the minimal distance,
//   key_hi = (2 p.c_k - |c_k|^2) * 512 + k         : ... the LARGEST.
// Both are dot * 1024 + a per-entry constant: per (pixel, entry) 1 IDP4A + 2 multiply/shift-adds, and a 3-input maximum
// takes two entries at a time.  |2 p.c - |c|^2| <= 390150 < 2^22, so the keys fit 32 bits.  Almost always the two
// indices agree (one entry at the minimum) and that is the answer; if they differ, every entry at the minimum lies
// between them and the reference's visiting order (start, +1, -1, +2, ...) decides among those.
constexpr int kIntColors = 512;
constexpr int kIntSentinel = -(1 << 30);  // pads an odd palette: loses against every real key (>= -2^27)

__device__ __forceinline__ void stage_palette_int(const uint32_t *sorted, int num_colors, int4 *s_ent) {
  const int padded = (num_colors + 1) & ~1;
  for (int k = threadIdx.x; k < padded; k += blockDim.x) {
    if (k < num_colors) {
      const uint32_t c = sorted[k] & 0x00FFFFFFu;
      const int r = (c >> 16) & 0xFF, g = (c >> 8) & 0xFF, b = c & 0xFF;
      const int sq = -(r * r + g * g + b * b) * 512;
      s_ent[k] = make_int4((int)c, sq + (511 - k), sq + k, (int)c);
    } else {
      s_ent[k] = make_int4(0, kIntSentinel, kIntSentinel, 0);
    }
  }
}

template <int PIX>
__device__ __forceinline__ void nearest_int(const int4 *s_ent, int num_colors, const uint32_t (&c)[PIX], int (&lo)[PIX], int (&hi)[PIX]) {
#pragma unroll
  for (int i = 0; i < PIX; ++i) lo[i] = hi[i] = kIntSentinel;
  const int padded = (num_colors + 1) & ~1;
#pragma unroll 4
  for (int k = 0; k < padded; k += 2) {
    const int4 e0 = s_ent[k], e1 = s_ent[k + 1];
#pragma unroll
    for (int i = 0; i < PIX; ++i) {
      const int d0 = (int)__dp4a(c[i], (uint32_t)e0.x, 0u) << 10, d1 = (int)__dp4a(c[i], (uint32_t)e1.x, 0u) << 10;
      lo[i] = max(lo[i], max(d0 + e0.y, d1 + e1.y));
      hi[i] = max(hi[i], max(d0 + e0.z, d1 + e1.z));
    }
  }
}

// The sorted-palette index of the entry one colour maps to, from its two keys; s = the reference's start index for it.
__device__ __forceinline__ int resolve_int_index(const int4 *s_ent, uint32_t c, int s, int lo, int hi) {
  const int ka = 511 - (lo & 511), kb = hi & 511;
  int win = ka;
  if (ka != kb) {
    // entries at the minimal distance: ka < ... < kb.  Above the start the rank grows with k, below it falls with k.
    if (s <= ka) {
      win = ka;
    } else if (s > kb) {
      win = kb;
    } else {
      const int want = lo >> 9;
      win = -1;
      for (int d = 0; win < 0; ++d) {
        const int up = s + d, down = s - d;
        if (up <= kb && ((((int)__dp4a(c, (uint32_t)s_ent[up].x, 0u) << 10) + s_ent[up].y) >> 9) == want) win = up;
        else if (d > 0 && down >= ka && ((((int)__dp4a(c, (uint32_t)s_ent[down].x, 0u) << 10) + s_ent[down].y) >> 9) == want) win = down;
      }
    }
  }
  return win;
}

// The palette word for one colour from its two keys.
__device__ __forceinline__ uint32_t resolve_int(const int4 *s_ent, uint32_t c, int s, int lo, int hi) {
  return (uint32_t)s_ent[resolve_int_index(s_ent, c, s, lo, hi)].w;
}

}  // namespace dq

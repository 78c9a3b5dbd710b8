// dq_hist_chunk.cuh -- hist_insert_chunked_kernel: the contiguous-sampling histogram of large inputs, counted per pixel
// chunk in shared memory before the L2 atomics.  Included by dq_hist.cu and by tools/microbench/hist_mb.cu (which times this very kernel), so
// it lives in one translation unit per binary.
//
// Every CTA owns contiguous chunks of `chunk_vec` uint4 (kChunk pixels; grid-stride over chunks).  A chunk spans
// several image rows, so it sees each colour of its neighbourhood many times: a G1 4K chunk of 32 768 pixels holds about
// 4 100 distinct colours.  The CTA counts them in an open-addressing table in shared memory (8 192 slots of 24-bit key
// + u32 count = 64 KB, linear probing) and at the end of the chunk adds each slot's count to the direct table with one
// L2 atomic, instead of one per pixel.  Results are the same integers as one atomic per pixel; only the order of the
// unique list changes, and that is the arrival order of atomics either way.
//
// Overflow: a colour that finds no slot within kMaxProbe probes takes the per-pixel global path, and once a chunk has
// put kFillMax keys into the table (incoherent input, e.g. uniform random pixels) every further pixel of that chunk does.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace dq {
namespace {

namespace hist_chunk {
constexpr int kThreads = 512;
constexpr int kVecPerThread = 2;                   // uint4 loads per thread and pass: 4 096 pixels per CTA pass
constexpr uint32_t kPassVec = kThreads * kVecPerThread;
constexpr uint32_t kSlotBits = 13;
constexpr uint32_t kSlots = 1u << kSlotBits;       // keys[kSlots], counts[kSlots]
constexpr uint32_t kChunk = 32768;                 // pixels per chunk: ~8x fewer L2 atomics than pixels on G1 4K
constexpr uint32_t kFillMax = kSlots * 5u / 8u;    // keys after which the rest of a chunk goes direct; checked every
                                                   // 4 pixels per thread, so the table stays below 7 168 keys
constexpr int kMaxProbe = 16;
constexpr uint32_t kEmpty = 0xFFFFFFFFu;           // keys are 24-bit colours
constexpr size_t kSmemBytes = (2 * (size_t)kSlots + 1) * sizeof(uint32_t);  // + the fill counter
}  // namespace hist_chunk

__device__ __forceinline__ uint32_t cut_colour(uint32_t pixel, uint32_t word_mask, uint32_t shift) {
  // whole-word variant of cut_bits (DivQuantUni.cpp:60-74); mask also drops the alpha byte
  return (pixel & word_mask) >> shift;
}

// seen_init (may be null): second direct table; a colour's entry is set to 0xFFFFFFFF by its first toucher, which is
// what the first-seen pass of the small-input path starts from (dq_split_exact.cu).
__device__ __forceinline__ void insert_colour(uint32_t c, bool active, uint32_t *table, uint32_t *uniq,
                                              uint32_t *ucount, uint32_t *seen_init) {
  bool fresh = false;
  if (active) fresh = (atomicAdd(table + c, 1u) == 0u);
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

// The colours whose table counter was 0 before this thread's atomic (old[k] == 0) go to the unique list: one cursor bump
// per warp.  Whole warps must call it.
template <int N>
__device__ __forceinline__ void append_fresh(const uint32_t (&c)[N], const uint32_t (&old)[N], uint32_t *uniq,
                                             uint32_t *ucount, uint32_t *seen_init) {
  unsigned m[N];
  unsigned any = 0;
  uint32_t total = 0;
#pragma unroll
  for (int k = 0; k < N; ++k) {
    m[k] = __ballot_sync(0xffffffffu, old[k] == 0u);
    any |= m[k];
    total += __popc(m[k]);
  }
  if (any) {
    const int lane = threadIdx.x & 31;
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(ucount, total);
    base = __shfl_sync(0xffffffffu, base, 0);
    const unsigned below = (1u << lane) - 1u;
#pragma unroll
    for (int k = 0; k < N; ++k) {
      if (old[k] == 0u) {
        uniq[base + __popc(m[k] & below)] = c[k];
        if (seen_init) seen_init[c[k]] = 0xFFFFFFFFu;
      }
      base += __popc(m[k]);
    }
  }
}

// count += 1 for colour c in the shared table; false when no slot was found within kMaxProbe probes.  In the steady
// state (key present at its home slot) this is one shared load and one shared atomic.
__device__ __forceinline__ bool count_shared(uint32_t c, uint32_t *keys, uint32_t *counts, uint32_t &inserted) {
  using namespace hist_chunk;
  uint32_t h = (c * 0x9E3779B1u) >> (32 - kSlotBits);
  for (int probe = 0; probe < kMaxProbe; ++probe) {
    uint32_t k = reinterpret_cast<volatile uint32_t *>(keys)[h];
    if (k == kEmpty) {
      k = atomicCAS(keys + h, kEmpty, c);
      if (k == kEmpty) {
        ++inserted;
        k = c;
      }
    }
    if (k == c) {
      atomicAdd(counts + h, 1u);
      return true;
    }
    h = (h + 1u) & (kSlots - 1u);
  }
  return false;
}

// Contiguous sampling (dec_factor == 1, numRows == 1: every live caller, quant_util.cpp:60) of inputs with at least one
// chunk per SM; smaller ones take the per-pixel hist_insert_kernel of dq_hist.cu.  Dynamic shared memory: kSmemBytes.
__global__ void __launch_bounds__(hist_chunk::kThreads, 2)
    hist_insert_chunked_kernel(const uint32_t *__restrict__ in, uint32_t n, uint32_t chunk_vec, uint32_t word_mask,
                               uint32_t shift, uint32_t *table, uint32_t *uniq, uint32_t *ucount, uint32_t *seen_init) {
  using namespace hist_chunk;
  extern __shared__ uint32_t hist_smem[];
  uint32_t *keys = hist_smem, *counts = hist_smem + kSlots, *fill = hist_smem + 2 * kSlots;
  for (uint32_t s = threadIdx.x; s < kSlots; s += kThreads) {
    keys[s] = kEmpty;
    counts[s] = 0u;
  }
  if (threadIdx.x == 0) *fill = 0u;
  __syncthreads();

  const uint32_t nvec = n >> 2;
  const uint4 *in4 = reinterpret_cast<const uint4 *>(in);
  const int lane = threadIdx.x & 31;
  for (uint32_t v0 = blockIdx.x * chunk_vec; v0 < nvec; v0 += gridDim.x * chunk_vec) {
    const uint32_t v1 = min(v0 + chunk_vec, nvec);
    // the loads of pass i + 1 are in flight while pass i is counted
    uint4 next[kVecPerThread];
#pragma unroll
    for (int j = 0; j < kVecPerThread; ++j) {
      const uint32_t i = v0 + j * kThreads + threadIdx.x;
      next[j] = i < v1 ? __ldcs(in4 + i) : make_uint4(0, 0, 0, 0);  // streamed once: keep L2 for the table
    }
    // whole CTAs iterate together so the ballots below are convergent
    for (uint32_t pass = v0; pass < v1; pass += kPassVec) {
      uint4 p[kVecPerThread];
#pragma unroll
      for (int j = 0; j < kVecPerThread; ++j) {
        p[j] = next[j];
        const uint32_t i = pass + kPassVec + j * kThreads + threadIdx.x;
        next[j] = i < v1 ? __ldcs(in4 + i) : make_uint4(0, 0, 0, 0);
      }
      uint32_t c[4 * kVecPerThread], old[4 * kVecPerThread];
      bool global = false;
#pragma unroll
      for (int j = 0; j < kVecPerThread; ++j) {
        const bool ok = pass + j * kThreads + threadIdx.x < v1;
        // a full table sends the rest of the chunk direct (the same for the whole warp)
        const bool direct = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t *>(fill), 0) >= kFillMax;
        uint32_t inserted = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int k = 4 * j + q;
          const uint32_t px = q == 0 ? p[j].x : q == 1 ? p[j].y : q == 2 ? p[j].z : p[j].w;
          c[k] = cut_colour(px, word_mask, shift);
          old[k] = (ok && (direct || !count_shared(c[k], keys, counts, inserted))) ? 0u : 1u;  // 0: needs the L2 atomic
          global |= old[k] == 0u;
        }
        if (!direct) {
          const uint32_t ins = __reduce_add_sync(0xffffffffu, inserted);
          if (lane == 0 && ins) atomicAdd(fill, ins);
        }
      }
      if (__any_sync(0xffffffffu, global)) {
        // all the pixel atomics are issued before any of their results is looked at
#pragma unroll
        for (int k = 0; k < 4 * kVecPerThread; ++k)
          if (old[k] == 0u) old[k] = atomicAdd(table + c[k], 1u);
        append_fresh(c, old, uniq, ucount, seen_init);
      }
    }
    // flush: one L2 atomic per distinct colour of the chunk, and the table is empty again for the next chunk
    __syncthreads();
#pragma unroll 1
    for (uint32_t s0 = 0; s0 < kSlots; s0 += 4 * kThreads) {
      uint32_t c[4], old[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t s = s0 + k * kThreads + threadIdx.x;
        c[k] = keys[s];
        old[k] = 1u;
        if (c[k] != kEmpty) {
          old[k] = atomicAdd(table + c[k], counts[s]);
          keys[s] = kEmpty;
          counts[s] = 0u;
        }
      }
      append_fresh(c, old, uniq, ucount, seen_init);
    }
    if (threadIdx.x == 0) *fill = 0u;
    __syncthreads();
  }
  // tail (< 4 pixels) handled by the first warp of the grid
  if (blockIdx.x == 0 && threadIdx.x < 32) {
    const uint32_t i = (nvec << 2) + threadIdx.x;
    const bool ok = i < n;
    const uint32_t p = ok ? in[i] : 0u;
    insert_colour(cut_colour(p, word_mask, shift), ok, table, uniq, ucount, seen_init);
  }
}

}  // namespace
}  // namespace dq

// Histogram variants on G1-like data (SURVEY 8d generator), 3840x2160: which formulation of the
// "count += 1 per pixel, list the unique colours" step is fastest on B200?
// The last section times the library's hist_insert_chunked_kernel (dq_hist_chunk.cuh: shared-memory counts per
// contiguous pixel chunk) for several chunk sizes, against the per-pixel kernel, on all SMs and on a grid of 48 CTAs (about what the frame
// pipeline leaves free), plus the raw rate of shared-memory atomics on hashed slots.
#include <cstdio>
#include <cstdint>
#include <algorithm>
#include <vector>
#include <cuda_runtime.h>
#include "dq_hist_chunk.cuh"
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA %s at %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)
__global__ void gen(uint32_t *px, int W, int H, int uniform = 0) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (size_t)W * H; i += (size_t)gridDim.x * blockDim.x) {
    int x = i % W, y = i / W;
    uint64_t s = 12345 + (i + 1) * 0x9E3779B97F4A7C15ull, z = s;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; z ^= z >> 31;
    if (uniform) { px[i] = 0xFF000000u | (uint32_t)(z >> 40); continue; }
    int n = (int)(z % 9) - 4;
    int r = min(255, max(0, x * 255 / W + n)), g = min(255, max(0, y * 255 / H + n)), b = min(255, max(0, (x + y) * 255 / (W + H) + n));
    px[i] = 0xFF000000u | (r << 16) | (g << 8) | b;
  }
}
__global__ void __launch_bounds__(256) k_atom_append(const uint4 *in, uint32_t nvec, uint32_t *table, uint32_t *uniq, uint32_t *ucount) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += gridDim.x * blockDim.x) {
    uint4 p = __ldcs(in + i); uint32_t c[4] = {p.x & 0xFFFFFF, p.y & 0xFFFFFF, p.z & 0xFFFFFF, p.w & 0xFFFFFF};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      bool fresh = atomicAdd(table + c[k], 1u) == 0u;
      unsigned m = __ballot_sync(0xffffffffu, fresh);
      if (m) { int lane = threadIdx.x & 31; uint32_t base = 0; if (lane == __ffs(m) - 1) base = atomicAdd(ucount, __popc(m)); base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1); if (fresh) uniq[base + __popc(m & ((1u << lane) - 1))] = c[k]; }
    }
  }
}
__global__ void __launch_bounds__(256) k_red(const uint4 *in, uint32_t nvec, uint32_t *table, unsigned char *flags) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += gridDim.x * blockDim.x) {
    uint4 p = __ldcs(in + i); uint32_t c[4] = {p.x & 0xFFFFFF, p.y & 0xFFFFFF, p.z & 0xFFFFFF, p.w & 0xFFFFFF};
#pragma unroll
    for (int k = 0; k < 4; ++k) { atomicAdd(table + c[k], 1u); if (flags) flags[c[k] >> 8] = 1; }
  }
}
// warp-merged: equal colours among the 32 lanes (pixel k of each thread) are counted by one lane
__global__ void __launch_bounds__(256) k_atom_match(const uint4 *in, uint32_t nvec, uint32_t *table, uint32_t *uniq, uint32_t *ucount) {
  const uint32_t nround = (nvec + 31u) & ~31u;
  const int lane = threadIdx.x & 31;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nround; i += gridDim.x * blockDim.x) {
    const bool ok = i < nvec;
    uint4 p = ok ? __ldcs(in + i) : make_uint4(0, 0, 0, 0);
    uint32_t c[4] = {p.x & 0xFFFFFF, p.y & 0xFFFFFF, p.z & 0xFFFFFF, p.w & 0xFFFFFF};
    uint32_t old[4] = {1u, 1u, 1u, 1u};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const unsigned m = __match_any_sync(0xffffffffu, ok ? c[k] : 0xFFFFFFFFu);
      if (ok && lane == __ffs(m) - 1) old[k] = atomicAdd(table + c[k], (uint32_t)__popc(m));
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      bool fresh = old[k] == 0u;
      unsigned m = __ballot_sync(0xffffffffu, fresh);
      if (m) { uint32_t base = 0; if (lane == __ffs(m) - 1) base = atomicAdd(ucount, __popc(m)); base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1); if (fresh) uniq[base + __popc(m & ((1u << lane) - 1))] = c[k]; }
    }
  }
}
// RED for the count + a 2 MB bitmap for "seen": a plain (cacheable) read filters the pixels whose colour is known
// already, only the others pay an atomicOr with return; the thread that flips the bit appends the colour.
__global__ void __launch_bounds__(256) k_red_bitmap(const uint4 *in, uint32_t nvec, uint32_t *table, uint32_t *bitmap, uint32_t *uniq, uint32_t *ucount) {
  const uint32_t nround = (nvec + 31u) & ~31u;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nround; i += gridDim.x * blockDim.x) {
    const bool ok = i < nvec;
    uint4 p = ok ? __ldcs(in + i) : make_uint4(0, 0, 0, 0);
    uint32_t c[4] = {p.x & 0xFFFFFF, p.y & 0xFFFFFF, p.z & 0xFFFFFF, p.w & 0xFFFFFF};
    uint32_t seen[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { if (ok) atomicAdd(table + c[k], 1u); seen[k] = ok ? bitmap[c[k] >> 5] : 0xFFFFFFFFu; }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t bit = 1u << (c[k] & 31);
      bool fresh = false;
      if (ok && !(seen[k] & bit)) fresh = !(atomicOr(bitmap + (c[k] >> 5), bit) & bit);
      unsigned m = __ballot_sync(0xffffffffu, fresh);
      if (m) { int lane = threadIdx.x & 31; uint32_t base = 0; if (lane == __ffs(m) - 1) base = atomicAdd(ucount, __popc(m)); base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1); if (fresh) uniq[base + __popc(m & ((1u << lane) - 1))] = c[k]; }
    }
  }
}
__global__ void clear_uniq_bitmap(uint32_t *table, uint32_t *bitmap, const uint32_t *uniq, const uint32_t *ucount) { for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < *ucount; i += gridDim.x * blockDim.x) { table[uniq[i]] = 0; bitmap[uniq[i] >> 5] = 0; } }
// neighbour-merged: equal colours among the 4 pixels of a thread are counted once
__global__ void __launch_bounds__(256) k_red_merge(const uint4 *in, uint32_t nvec, uint32_t *table) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += gridDim.x * blockDim.x) {
    uint4 p = __ldcs(in + i); uint32_t c[4] = {p.x & 0xFFFFFF, p.y & 0xFFFFFF, p.z & 0xFFFFFF, p.w & 0xFFFFFF};
    uint32_t n[4] = {1, 1, 1, 1};
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b2 = a + 1; b2 < 4; ++b2) if (n[b2] && c[b2] == c[a] && n[a]) { n[a] += n[b2]; n[b2] = 0; }
#pragma unroll
    for (int k = 0; k < 4; ++k) if (n[k]) atomicAdd(table + c[k], n[k]);
  }
}
// scan of flagged 256-entry blocks: emit (colour,count), clear the table
__global__ void __launch_bounds__(256) k_scan(uint32_t *table, unsigned char *flags, uint2 *pts, uint32_t *ucount) {
  const int lane = threadIdx.x & 31;
  for (uint32_t blk = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32; blk < 65536; blk += gridDim.x * (blockDim.x / 32)) {
    if (!flags[blk]) continue;
    if (lane == 0) flags[blk] = 0;
    for (int j = 0; j < 8; ++j) {
      uint32_t c = blk * 256 + j * 32 + lane; uint32_t v = table[c];
      unsigned m = __ballot_sync(0xffffffffu, v != 0);
      if (m) { uint32_t base = 0; if (lane == 0) base = atomicAdd(ucount, __popc(m)); base = __shfl_sync(0xffffffffu, base, 0);
        if (v) { pts[base + __popc(m & ((1u << lane) - 1))] = make_uint2(c, v); table[c] = 0; } }
    }
  }
}
__global__ void clear_uniq(uint32_t *table, const uint32_t *uniq, const uint32_t *ucount) { for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < *ucount; i += gridDim.x * blockDim.x) table[uniq[i]] = 0; }

// the library's per-pixel hist_insert_kernel (4 L2 atomics in flight per thread)
__global__ void __launch_bounds__(256) k_direct4(const uint4 *in4, uint32_t nvec, uint32_t *table, uint32_t *uniq, uint32_t *ucount) {
  const uint32_t nround = (nvec + 31u) & ~31u;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nround; i += gridDim.x * blockDim.x) {
    const bool ok = i < nvec;
    uint4 p = ok ? __ldcs(in4 + i) : make_uint4(0, 0, 0, 0);
    uint32_t c[4] = {p.x & 0xFFFFFF, p.y & 0xFFFFFF, p.z & 0xFFFFFF, p.w & 0xFFFFFF};
    uint32_t old[4] = {1u, 1u, 1u, 1u};
    if (ok) {
#pragma unroll
      for (int k = 0; k < 4; ++k) old[k] = atomicAdd(table + c[k], 1u);
    }
    dq::append_fresh(c, old, uniq, ucount, nullptr);
  }
}
// shared-memory atomics on 8192 slots: hashed slots (bank conflicts as a hash gives them) or one bank per lane
__global__ void __launch_bounds__(512) k_smem_atom(uint32_t iters, uint32_t *sink, int cas, int per_lane_bank) {
  __shared__ uint32_t t[8192];
  for (int s = threadIdx.x; s < 8192; s += blockDim.x) t[s] = 0;
  __syncthreads();
  uint32_t h = threadIdx.x * 0x9E3779B1u + blockIdx.x * 7919u, acc = 0;
  for (uint32_t i = 0; i < iters; ++i) {
    h = h * 1664525u + 1013904223u;
    uint32_t slot = h >> 19;
    if (per_lane_bank) slot = (slot & ~31u) | (threadIdx.x & 31);
    if (cas) acc ^= atomicCAS(t + slot, i, i + 1u); else atomicAdd(t + slot, 1u);
  }
  __syncthreads();
  if (threadIdx.x == 0) sink[blockIdx.x] = t[0] + acc;
}
static float median(std::vector<float> v) { std::sort(v.begin(), v.end()); return v[v.size() / 2]; }
// time `launch` (median of 7), clearing the direct table after each run; prints U of the last run
template <class F>
static float time_hist(F launch, uint32_t *table, uint32_t *uniq, uint32_t *ucount, uint32_t *u_out) {
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  std::vector<float> t;
  for (int rep = 0; rep < 8; ++rep) {
    cudaMemset(ucount, 0, 4); cudaEventRecord(e0); launch(); cudaEventRecord(e1); cudaDeviceSynchronize();
    float ms; cudaEventElapsedTime(&ms, e0, e1); if (rep) t.push_back(ms);
    cudaMemcpy(u_out, ucount, 4, cudaMemcpyDeviceToHost);
    clear_uniq<<<592, 256>>>(table, uniq, ucount); cudaDeviceSynchronize();
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return median(t) * 1e3f;
}
static int chunked_section(uint32_t *px, uint32_t *table, uint32_t *uniq, uint32_t *ucount) {
  int sms = 0; CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
  CK(cudaFuncSetAttribute(dq::hist_insert_chunked_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dq::hist_chunk::kSmemBytes));
  {
    uint32_t *sink; CK(cudaMalloc(&sink, 4096 * 4));
    const int grid = 2 * sms; const uint32_t iters = 8192;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int cas = 0; cas < 2; ++cas)
      for (int bank = 0; bank < 2; ++bank) {
        std::vector<float> t;
        for (int rep = 0; rep < 5; ++rep) {
          cudaEventRecord(e0); k_smem_atom<<<grid, 512>>>(iters, sink, cas, bank); cudaEventRecord(e1); CK(cudaDeviceSynchronize());
          float ms; cudaEventElapsedTime(&ms, e0, e1); if (rep) t.push_back(ms);
        }
        const double ops = (double)grid * 512 * iters, ms = median(t);
        printf("shared %-9s %-16s: %.1f G/s device-wide, %.2f per SM per clock-ns\n", cas ? "atomicCAS" : "atomicAdd",
               bank ? "one bank / lane" : "hashed slots", ops / (ms * 1e6), ops / (ms * 1e6) / sms);
      }
  }
  struct In { const char *name; int W, H, uniform; };
  for (In in : {In{"G1 3840x2160", 3840, 2160, 0}, In{"G1 1920x1080", 1920, 1080, 0}, In{"G2 1920x1080", 1920, 1080, 1}}) {
    const uint32_t N = (uint32_t)in.W * in.H;
    gen<<<1184, 256>>>(px, in.W, in.H, in.uniform); CK(cudaDeviceSynchronize());
    uint32_t u = 0;
    for (int grid : {8 * sms, 96, 48}) {
      const float us = time_hist([&] { k_direct4<<<grid, 256>>>((const uint4 *)px, N / 4, table, uniq, ucount); }, table, uniq, ucount, &u);
      printf("%s per-pixel kernel          grid %4d x 256: %6.1f us  U=%u\n", in.name, grid, us, u);
    }
    for (uint32_t chunk : {16384u, 32768u, 65536u}) {
      const int all = (int)std::min<uint32_t>((N + chunk - 1) / chunk, 8u * sms);
      for (int grid : {all, 48}) {
        const float us = time_hist([&] {
          dq::hist_insert_chunked_kernel<<<grid, dq::hist_chunk::kThreads, dq::hist_chunk::kSmemBytes>>>(px, N, chunk / 4, 0x00FFFFFFu, 0u,
                                                                                               table, uniq, ucount, nullptr);
        }, table, uniq, ucount, &u);
        printf("%s chunked kernel chunk %5u grid %4d x 512: %6.1f us  U=%u%s\n", in.name, chunk, grid, us, u,
               chunk == dq::hist_chunk::kChunk && grid == all && N / chunk >= (uint32_t)sms ? "  <- library's choice" : "");
      }
    }
    CK(cudaGetLastError());
  }
  return 0;
}
int main() {
  const int W = 3840, H = 2160; const uint32_t N = W * H;
  uint32_t *px, *table, *uniq, *ucount; unsigned char *flags; uint2 *pts;
  CK(cudaMalloc(&px, N * 4)); CK(cudaMalloc(&table, 64 << 20)); CK(cudaMalloc(&uniq, N * 4)); CK(cudaMalloc(&ucount, 4)); CK(cudaMalloc(&flags, 65536)); CK(cudaMalloc(&pts, (size_t)N * 8));
  CK(cudaMemset(table, 0, 64 << 20)); CK(cudaMemset(flags, 0, 65536));
  gen<<<1184, 256>>>(px, W, H); CK(cudaDeviceSynchronize());
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1); float ms;
  for (int grid : {1184, 2368, 4736}) {
    for (int rep = 0; rep < 3; ++rep) {
      CK(cudaMemset(ucount, 0, 4)); cudaEventRecord(e0);
      k_atom_append<<<grid, 256>>>((uint4 *)px, N / 4, table, uniq, ucount);
      cudaEventRecord(e1); CK(cudaDeviceSynchronize()); cudaEventElapsedTime(&ms, e0, e1);
      uint32_t u; CK(cudaMemcpy(&u, ucount, 4, cudaMemcpyDeviceToHost));
      if (rep == 2) printf("atom+append  grid %5d: %.1f us  U=%u\n", grid, ms * 1e3, u);
      clear_uniq<<<592, 256>>>(table, uniq, ucount); CK(cudaDeviceSynchronize());
    }
  }
  for (int grid : {1184, 2368}) {
    for (int rep = 0; rep < 3; ++rep) {
      CK(cudaMemset(ucount, 0, 4)); cudaEventRecord(e0);
      k_atom_match<<<grid, 256>>>((uint4 *)px, N / 4, table, uniq, ucount);
      cudaEventRecord(e1); CK(cudaDeviceSynchronize()); cudaEventElapsedTime(&ms, e0, e1);
      uint32_t u; CK(cudaMemcpy(&u, ucount, 4, cudaMemcpyDeviceToHost));
      if (rep == 2) printf("atom+match   grid %5d: %.1f us  U=%u\n", grid, ms * 1e3, u);
      clear_uniq<<<592, 256>>>(table, uniq, ucount); CK(cudaDeviceSynchronize());
    }
  }
  {
    uint32_t *bitmap; CK(cudaMalloc(&bitmap, 2 << 20)); CK(cudaMemset(bitmap, 0, 2 << 20));
    for (int grid : {1184, 2368, 4736}) {
      for (int rep = 0; rep < 3; ++rep) {
        CK(cudaMemset(ucount, 0, 4)); cudaEventRecord(e0);
        k_red_bitmap<<<grid, 256>>>((uint4 *)px, N / 4, table, bitmap, uniq, ucount);
        cudaEventRecord(e1); CK(cudaDeviceSynchronize()); cudaEventElapsedTime(&ms, e0, e1);
        uint32_t u; CK(cudaMemcpy(&u, ucount, 4, cudaMemcpyDeviceToHost));
        if (rep == 2) printf("RED+bitmap   grid %5d: %.1f us  U=%u\n", grid, ms * 1e3, u);
        clear_uniq_bitmap<<<592, 256>>>(table, bitmap, uniq, ucount); CK(cudaDeviceSynchronize());
      }
    }
  }
  for (int withflags = 0; withflags < 2; ++withflags) {
    for (int rep = 0; rep < 3; ++rep) {
      CK(cudaMemset(ucount, 0, 4)); cudaEventRecord(e0);
      k_red<<<2368, 256>>>((uint4 *)px, N / 4, table, withflags ? flags : nullptr);
      cudaEventRecord(e1); CK(cudaDeviceSynchronize()); cudaEventElapsedTime(&ms, e0, e1);
      float ms1 = ms;
      if (!withflags) CK(cudaMemset(flags, 1, 65536));
      cudaEventRecord(e0); k_scan<<<1184, 256>>>(table, flags, pts, ucount); cudaEventRecord(e1); CK(cudaDeviceSynchronize()); cudaEventElapsedTime(&ms, e0, e1);
      uint32_t u; CK(cudaMemcpy(&u, ucount, 4, cudaMemcpyDeviceToHost));
      if (rep == 2) printf("RED%s: %.1f us ; scan+clear (%s): %.1f us  U=%u\n", withflags ? "+flags" : "      ", ms1 * 1e3, withflags ? "flagged blocks" : "all 16M bins", ms * 1e3, u);
    }
  }
  for (int rep = 0; rep < 3; ++rep) {
    cudaEventRecord(e0); k_red_merge<<<2368, 256>>>((uint4 *)px, N / 4, table); cudaEventRecord(e1); CK(cudaDeviceSynchronize()); cudaEventElapsedTime(&ms, e0, e1);
    if (rep == 2) printf("RED neighbour-merged: %.1f us\n", ms * 1e3);
    CK(cudaMemset(table, 0, 64 << 20));
  }
  return chunked_section(px, table, uniq, ucount);
}

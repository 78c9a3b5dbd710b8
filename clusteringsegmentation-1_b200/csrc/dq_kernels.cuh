// dq_kernels.cuh -- host-callable launchers of the histogram and remap kernels.
#pragma once

#include "dq_common.cuh"

namespace dq {

// ---- dq_hist.cu ----
void hist_insert(const uint32_t *d_in, uint32_t n, uint32_t num_rows, uint32_t num_cols, uint32_t dec, int num_bits,
                 uint32_t *d_table, uint32_t *d_uniq, uint32_t *d_ucount, int sm_count, cudaStream_t st,
                 uint32_t *d_seen_init = nullptr);
void hist_collect(const uint32_t *d_uniq, const uint32_t *d_ucount, uint32_t u_hint, uint32_t *d_table, uint2 *d_pts,
                  bool clear_table, int sm_count, cudaStream_t st);
void table_clear(const uint32_t *d_uniq, const uint32_t *d_ucount, uint32_t u_hint, uint32_t *d_table, int sm_count,
                 cudaStream_t st);
void points_from_pixels(const uint32_t *d_in, uint32_t n, uint2 *d_pts, int sm_count, cudaStream_t st);
void cut_bits_device(const uint32_t *d_in, uint32_t n, uint32_t *d_out, int rbits, int gbits, int bbits, int sm_count,
                     cudaStream_t st);
void order_keys(const uint32_t *d_in, uint32_t num_rows, uint32_t num_cols, uint32_t dec, int num_bits, const uint32_t *d_uniq,
                const uint2 *d_pts, uint32_t u, uint32_t *d_table, uint64_t *d_keys, int sm_count, cudaStream_t st);

// Sorts the u (unique) keys of order_keys with their point index (d_keys / d_vals need room for the next power of two),
// then writes the unique colours and their weights norm * count in that order: calc_color_table's output, on the device.
void order_sort(uint64_t *d_keys, uint32_t *d_vals, uint32_t u, int sm_count, cudaStream_t st);
void order_sort_emit(const uint2 *d_pts, uint32_t u, uint64_t *d_keys, uint32_t *d_vals, double norm, uint32_t *d_colours,
                     double *d_weights, int sm_count, cudaStream_t st);
void hist_export(const uint2 *d_pts, const uint32_t *d_ucount, uint32_t u_hint, uint32_t *d_colours, uint32_t *d_counts,
                 int sm_count, cudaStream_t st);
// d_first (optional, cap + 1 words): the shard-local first-seen index of every exported colour (from d_first_table), then
// n_shard
void hist_export_padded(const uint2 *d_pts, const uint32_t *d_ucount, uint32_t cap, uint32_t *d_colours, uint32_t *d_counts,
                        uint32_t *d_overflow, int sm_count, cudaStream_t st, const uint32_t *d_first_table = nullptr,
                        uint32_t *d_first = nullptr, uint32_t n_shard = 0);
void hist_merge(const uint32_t *d_colours, const uint32_t *d_counts, uint32_t num_entries, uint32_t *d_table, uint32_t *d_uniq,
                uint32_t *d_ucount, int sm_count, cudaStream_t st, uint32_t *d_seen_init = nullptr);
// After hist_merge with d_seen_init = d_first_seen: the whole image's first-seen index of every merged colour (exported
// lists [world][cap], first-seen slices [world][cap + 1] as hist_export_padded writes them)
void hist_merge_first(const uint32_t *d_colours, const uint32_t *d_counts, const uint32_t *d_first, uint32_t cap, uint32_t world,
                      uint32_t *d_first_seen, int sm_count, cudaStream_t st);

// ---- dq_map.cu ----
int map_smem_palette_limit();
void map_pixels(const uint32_t *d_in, uint32_t n, uint32_t *d_out, const uint32_t *d_sorted, int num_colors,
                const int *d_lut, int4 *d_pal_scratch, int sm_count, cudaStream_t st);
void map_unique(const uint32_t *d_uniq, const uint32_t *d_ucount, uint32_t u_hint, uint32_t *d_table,
                const uint32_t *d_sorted, int num_colors, const int *d_lut, int sm_count, cudaStream_t st);
// Sorted palette and start-index table small enough (K <= 256) to travel inside the kernel's parameter block: no
// upload, no extra dependency between the host's table building and the launch.
struct MapTablesParam {
  uint32_t sorted[256];
  uint16_t lut[768];  // lut_init[0..765], values < K
};
void map_unique_params(const MapTablesParam &tables, const uint32_t *d_uniq, const uint32_t *d_ucount, uint32_t u_hint,
                       uint32_t *d_table, int num_colors, int sm_count, cudaStream_t st);
void block_vote(const uint32_t *d_quant, uint32_t width, uint32_t height, uint32_t dim, uint32_t *d_blocks, int sm_count,
                cudaStream_t st);
void map_labels(const uint32_t *d_in, uint32_t n, uint32_t *d_out, const uint2 *d_pairs, int num_pairs, int greyscale,
                uint32_t *d_error, int sm_count, cudaStream_t st);
void map_gather(const uint32_t *d_in, uint32_t n, uint32_t *d_out, const uint32_t *d_table, int sm_count, cudaStream_t st);

// ---- dq_srm.cu ----
uint32_t srm_num_pairs(uint32_t width, uint32_t height);
size_t srm_scratch_words(uint32_t width, uint32_t height);
// Returns the number of kernels launched.  d_pairs: 3 words per edge (r1, r2, diff) in merge order.
int srm_sorted_edges(const uint8_t *d_in, uint32_t width, uint32_t height, uint32_t channels, uint32_t width_step,
                     uint32_t *d_pairs, uint32_t *d_scratch, cudaStream_t st);

}  // namespace dq

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
// d_pal_scratch: num_colors int4 entries, used above map_smem_palette_limit() (as by map_pixels)
void map_unique(const uint32_t *d_uniq, const uint32_t *d_ucount, uint32_t u_hint, uint32_t *d_table,
                const uint32_t *d_sorted, int num_colors, const int *d_lut, int4 *d_pal_scratch, int sm_count, cudaStream_t st);
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

// ---- dq_batch.cu: quant_recurse over many small items (one CTA per item) ----
constexpr uint32_t kBatchMaxPoints = 4096;       // distinct colours a batched item may have (its points stay in shared memory)
constexpr uint32_t kBatchOverflow = 0xFFFFFFFFu;  // result word 0 of an item with more colours than that
constexpr uint32_t kBatchResultWords = 16;        // per item: [0] U | [1] palette entries [2] empty clusters | [4, 16) ctl words
constexpr int kBatchTilePixels = 1024;            // pixels per CTA of the remap
constexpr int kBatchLutEntries = 3 * 255 + 1;
struct BatchItem {
  uint32_t begin, n;  // pixels [begin, begin + n) of the flat input; the item's histogram slices start at begin as well
  uint32_t k, pal;    // requested K; offset of its palette in the palette buffer
};
struct BatchTile {
  uint32_t begin, end;  // pixels of the flat input
  uint32_t table;       // batched item whose tables map them
  uint32_t pad;
};
// One launch each, one CTA per item.  d_colours / d_counts / d_first: as many words as the flat input.
void batch_hist_launch(const uint32_t *d_in, const BatchItem *d_items, uint32_t num_items, uint32_t *d_colours, uint32_t *d_counts,
                       uint32_t *d_first, uint32_t *d_res, cudaStream_t st);
// Items whose U (result word 0) exceeds max_points (at most kBatchMaxPoints) are left alone.  d_cluster_size / d_cluster_mean:
// 1 / 3 entries per palette word.
void batch_split_launch(const BatchItem *d_items, uint32_t num_items, uint32_t max_points, const uint32_t *d_colours, uint32_t *d_counts,
                        const uint32_t *d_first, uint32_t *d_res, uint32_t *d_palette, uint32_t *d_cluster_size, double *d_cluster_mean,
                        cudaStream_t st);
// d_tables[i] = (offset in d_sorted, palette size) of batched item i, d_luts[i * kBatchLutEntries ...] its lut_init.
// d_labels != nullptr: also d_labels[p] = d_label_tables[offset + w] for the sorted entry w that pixel p maps to.
void batch_remap_launch(const uint32_t *d_in, uint32_t *d_out, const BatchTile *d_tiles, uint32_t num_tiles, const uint32_t *d_sorted,
                        const uint2 *d_tables, const uint16_t *d_luts, const uint16_t *d_label_tables, uint32_t *d_labels,
                        cudaStream_t st);

// ---- dq_srm.cu ----
// The stable counting sorts over tiles (SRM's edges, dq_regions.cu's tags) run 256 threads a CTA, one per bin.
constexpr int kSortThreads = 256;
// counts[bin][0 .. num_tiles) of num_bins bins: every row scanned (exclusive) in place, its total to row_total[bin]
void tile_rowscan_launch(uint32_t num_bins, uint32_t num_tiles, uint32_t *counts, uint32_t *row_total, cudaStream_t st);
uint32_t srm_num_pairs(uint32_t width, uint32_t height);
size_t srm_scratch_words(uint32_t width, uint32_t height);
// Returns the number of kernels launched.  d_pairs: 3 words per edge (r1, r2, diff) in merge order.
int srm_sorted_edges(const uint8_t *d_in, uint32_t width, uint32_t height, uint32_t channels, uint32_t width_step,
                     uint32_t *d_pairs, uint32_t *d_scratch, cudaStream_t st);

// ---- dq_regions.cu: stable partition of a tag image by region (dq_quant_regions_*, dq_map_regions_*) ----
uint32_t region_passes(uint32_t num_regions);  // digit passes of the sort: 1 up to 256 regions, 2 up to 65 536, 3 above
// d_scratch words for n pixels (n >= 1): per-tile digit counts, digit totals, the num_regions + 1 region offsets
size_t region_scratch_words(uint32_t n, uint32_t num_regions);
// Sorts the pixels with tags[p] < num_regions by tag, stable, in d_pairs (2 n pairs, ping-pong); *d_sorted = the m sorted
// (tag, index) pairs, d_gathered[j] = d_in[index of pair j], region_offsets(d_scratch, n) = num_regions + 1 offsets of the
// regions in that order (the last is m).  d_dropped: nullptr, or a bitmap of (num_regions + 31) / 32 words whose set bits
// mark regions whose pixels are dropped like those in no region.  Returns the number of kernels launched.
int region_partition(const uint32_t *d_in, const uint32_t *d_tags, uint32_t n, uint32_t num_regions, const uint32_t *d_dropped,
                     uint2 *d_pairs, uint32_t *d_gathered, uint32_t *d_scratch, const uint2 **d_sorted, cudaStream_t st);
const uint32_t *region_offsets(const uint32_t *d_scratch, uint32_t n);
// d_out[index of pair j] = d_g_out[j] and, with d_labels, d_labels[index] = d_g_labels[j] for j < m (one launch)
void region_scatter_back(const uint2 *d_sorted, uint32_t m, const uint32_t *d_g_out, const uint32_t *d_g_labels, uint32_t *d_out,
                         uint32_t *d_labels, cudaStream_t st);

}  // namespace dq

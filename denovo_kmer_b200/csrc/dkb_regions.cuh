// dkb_regions.cuh — region mode (DESIGN.md §2 "region-scoped counting"): the per-batch
// read-locus index that lets stage C of the scan resolve a verified seed to its read, and the
// per-entry copy of the variant windows its gate tests against.
#pragma once
#include "dkb_device.cuh"

namespace dkb {

// One thread per read: its first stream position (offsets[r] - offsets[0] + r, as the packer
// lays the batch out) and its alignment interval, an empty one normalised to {lo, 0}.
__global__ void k_read_loci(const uint64_t *offsets, const uint64_t *lo, const uint64_t *hi, uint32_t n_reads,
                            uint32_t *read_start, ulonglong2 *read_span) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  read_start[r] = (uint32_t)(offsets[r] - offsets[0]) + r;
  const uint64_t a = lo[r], b = hi[r];
  read_span[r] = make_ulonglong2(a, a < b ? b : 0ull);
}

// One thread per 2048-position tile (and one more): the last read that starts at or before
// the tile's first position, i.e. the first read that reaches into the tile.  Entry n_tiles
// is n_reads - 1, the upper end of the search for the last tile.
__global__ void k_tile_reads(const uint32_t *read_start, uint32_t n_reads, uint32_t n_tiles, uint32_t *tile_read) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n_tiles) return;
  if (t == n_tiles) {
    tile_read[t] = n_reads - 1;
    return;
  }
  const uint64_t p = (uint64_t)t << LOCI_TILE_SHIFT;
  uint32_t a = 0, b = n_reads - 1;  // read_start[0] == 0 <= p
  while (a < b) {
    const uint32_t mid = b - (b - a) / 2;
    if (read_start[mid] <= p) a = mid; else b = mid - 1;
  }
  tile_read[t] = a;
}

// One thread per entry: its variant's window, an empty one normalised to {lo, 0}.
__global__ void k_entry_windows(const uint32_t *variant, const ulonglong2 *var_win, uint32_t n_entries,
                                ulonglong2 *entry_win) {
  const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_entries) return;
  const ulonglong2 w = var_win[variant[e]];
  entry_win[e] = make_ulonglong2(w.x, w.x < w.y ? w.y : 0ull);
}

}  // namespace dkb

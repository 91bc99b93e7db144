// dkb_regions.cuh — region mode (DESIGN.md §2 "region-scoped counting"): the per-batch
// read-locus index that lets stage C of the scan resolve a verified seed to its read, and the
// per-entry copy of the variant windows its gate tests against.
#pragma once
#include "dkb_device.cuh"

namespace dkb {

// The segments of one launch's read-locus index: segment i holds reads [read_base[i],
// read_base[i + 1]) and tile hints [tile_base[i], tile_base[i + 1]) (its n_tiles + 1 entries).
// Its offsets are the batch's n_reads + 1, at read_base[i] + i of the concatenated offsets.
struct LociSegments {
  uint32_t n_seg;
  uint32_t read_base[MAX_SEGMENTS + 1];
  uint32_t tile_base[MAX_SEGMENTS + 1];
};

__device__ __forceinline__ uint32_t loci_segment(const uint32_t (&base)[MAX_SEGMENTS + 1], uint32_t n_seg,
                                                 uint32_t x) {
  uint32_t i = 0;
  while (i + 1 < n_seg && x >= base[i + 1]) i++;
  return i;
}

// One thread per read: its first stream position inside its segment (offsets[r] - offsets[0] +
// r, as the packer lays the batch out) and its alignment interval, an empty one normalised to
// {lo, 0}.
__global__ void k_read_loci(const LociSegments S, const uint64_t *offsets, const uint64_t *lo, const uint64_t *hi,
                            uint32_t *read_start, ulonglong2 *read_span) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= S.read_base[S.n_seg]) return;
  const uint32_t i = loci_segment(S.read_base, S.n_seg, r), q = r - S.read_base[i];
  const uint64_t *const off = offsets + S.read_base[i] + i;
  read_start[r] = (uint32_t)(off[q] - off[0]) + q;
  const uint64_t a = lo[r], b = hi[r];
  read_span[r] = make_ulonglong2(a, a < b ? b : 0ull);
}

// One thread per 2048-position tile of a segment (and one more): the last read of the segment
// that starts at or before the tile's first position, i.e. the first read that reaches into the
// tile.  The extra entry is the segment's last read, the upper end of the search for its last tile.
__global__ void k_tile_reads(const LociSegments S, const uint32_t *read_start, uint32_t *tile_read) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= S.tile_base[S.n_seg]) return;
  const uint32_t i = loci_segment(S.tile_base, S.n_seg, g), t = g - S.tile_base[i];
  const uint32_t first = S.read_base[i], last = S.read_base[i + 1] - 1;
  if (g + 1 == S.tile_base[i + 1]) {
    tile_read[g] = last;
    return;
  }
  const uint64_t p = (uint64_t)t << LOCI_TILE_SHIFT;
  uint32_t a = first, b = last;  // read_start[first] == 0 <= p
  while (a < b) {
    const uint32_t mid = b - (b - a) / 2;
    if (read_start[mid] <= p) a = mid; else b = mid - 1;
  }
  tile_read[g] = a;
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

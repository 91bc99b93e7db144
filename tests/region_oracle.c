/*
 * region_oracle.c — CPU restatement of region-scoped counting (DESIGN.md §2), test
 * infrastructure only.  orc_count_stream_loci is oracle/dnk_oracle.c's orc_count_stream with
 * the read index and the two window arrays: it walks the packed stream read by read (read r's
 * first base at stream position offsets[r] - offsets[0] + r) and counts a window toward entry e
 * only if read r's interval [rlo[r], rhi[r]) overlaps the window [vlo[v], vhi[v]) of e's
 * variant v, both non-empty.  Written the plain way and sharing nothing with the CUDA path;
 * tests/region_oracle.py pins it against a per-variant read fetch in pure Python.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define NO_ENTRY 0xFFFFFFFFu

typedef struct {
  uint64_t key;
  uint32_t ent;
} slot_t;

static size_t hash_key(uint64_t x, size_t cap) {
  x ^= x >> 33;
  x *= 0xFF51AFD7ED558CCDull;
  x ^= x >> 33;
  return (size_t)x & (cap - 1);
}

/* counts[n_entries] is ADDED to.  A repeated (key, variant, allele) triple keeps its first
 * entry live; later repeats stay at 0.  Returns 0, or -1 if memory runs out. */
int orc_count_stream_loci(const uint64_t *keys, const uint32_t *variant, const uint8_t *allele,
                          size_t n_entries, const uint64_t *vlo, const uint64_t *vhi,
                          const uint32_t *bases2, const uint32_t *mask1, uint64_t n_positions,
                          const uint64_t *offsets, const uint64_t *rlo, const uint64_t *rhi,
                          size_t n_reads, int k, uint64_t *counts, int n_threads) {
  size_t cap = 16;
  while (cap < 2 * n_entries + 2) cap <<= 1;
  slot_t *slots = (slot_t *)malloc(cap * sizeof(slot_t));
  if (!slots) return -1;
  for (size_t i = 0; i < cap; i++) slots[i].ent = NO_ENTRY;
  for (size_t i = 0; i < n_entries; i++) {
    size_t h = hash_key(keys[i], cap);
    int dup = 0;
    while (slots[h].ent != NO_ENTRY) {
      const uint32_t e = slots[h].ent;
      if (slots[h].key == keys[i] && variant[e] == variant[i] && allele[e] == allele[i]) dup = 1;
      h = (h + 1) & (cap - 1);
    }
    if (!dup) {
      slots[h].key = keys[i];
      slots[h].ent = (uint32_t)i;
    }
  }
  const uint64_t mask = (1ull << (2 * k)) - 1;
#ifdef _OPENMP
  if (n_threads < 1) n_threads = omp_get_max_threads();
#else
  n_threads = 1;
#endif
#pragma omp parallel for schedule(dynamic, 4096) num_threads(n_threads)
  for (long long r = 0; r < (long long)n_reads; r++) {
    const uint64_t a = rlo[r], b = rhi[r];
    if (a >= b) continue; /* unmapped: counts toward nothing */
    const uint64_t start = offsets[r] - offsets[0] + (uint64_t)r;
    const uint64_t end = start + (offsets[r + 1] - offsets[r]);
    uint64_t fwd = 0, rc = 0;
    int run = 0;
    for (uint64_t p = start; p < end && p < n_positions; p++) {
      if (!((mask1[p >> 5] >> (p & 31)) & 1u)) {
        run = 0;
        fwd = rc = 0;
        continue;
      }
      const uint64_t c = (bases2[p >> 4] >> (2 * (p & 15))) & 3u;
      fwd = ((fwd << 2) | c) & mask;
      rc = (rc >> 2) | ((3 - c) << (2 * (k - 1)));
      if (++run < k) continue;
      const uint64_t key = fwd < rc ? fwd : rc;
      for (size_t h = hash_key(key, cap); slots[h].ent != NO_ENTRY; h = (h + 1) & (cap - 1)) {
        if (slots[h].key != key) continue;
        const uint32_t e = slots[h].ent, v = variant[e];
        if (vlo[v] < vhi[v] && a < vhi[v] && vlo[v] < b) {
#pragma omp atomic
          counts[e]++;
        }
      }
    }
  }
  free(slots);
  return 0;
}

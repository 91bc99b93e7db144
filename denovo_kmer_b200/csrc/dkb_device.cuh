// dkb_device.cuh — device-side data layout and helpers shared by the build,
// scan and finalise kernels (sm_100a).  See DESIGN.md §3 for the layout.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dkb {

constexpr unsigned FULL_MASK = 0xffffffffu;

// ---- scan geometry -------------------------------------------------------
constexpr int SCAN_THREADS = 1024;         // one CTA per SM (shared-memory bound)
constexpr int SCAN_WARPS = SCAN_THREADS / 32;
constexpr int CHUNK = 64;                  // stream positions per lane per tile (4 words)
constexpr int WTILE = 32 * CHUNK;          // positions per warp tile (512 B of bases)
constexpr int WTILE_WORDS = WTILE / 16;    // 128 uint32 words of bases per warp tile
constexpr int BLOOM_WORDS = 51712;         // 202 KB seed filter resident in shared memory
// per-warp list of the filter-hit ids of one (macro) tile; denser tiles take several passes.
// Behind the pre-filter (mode 2) a macro tile has a handful of hits: 32 ids do, and the 6 KB go
// to the pre-filter instead (configs[1] 7.09 -> 7.23 Tbases/s; k = 21 at stride 8 4.14 -> 4.04).
constexpr int HL_CAP_WIDE = 128, HL_CAP_PRE = 32;
// Filter modes of the scan kernel (template parameter FM):
//   0 seed filter in shared memory      1 in L2      2 in L2 behind the shared-memory pre-filter
//   3, 4 = 1, 2 with GATED lookups: stage A also reads the flag stream and skips every lookup
//   whose seed holds an unusable base (no countable window can contain such a seed).  Saves the
//   lookup's load-path work, costs instructions: pays where the gathers bound the kernel.
__host__ __device__ constexpr bool fm_pre(int fm) { return fm == 2 || fm == 4; }
__host__ __device__ constexpr bool fm_gate(int fm) { return fm >= 3; }
__host__ __device__ constexpr int hl_cap(int fm) { return fm_pre(fm) ? HL_CAP_PRE : HL_CAP_WIDE; }
constexpr int CQ_CAP = 64;                 // per-warp ring of verified seeds
constexpr size_t scan_lists_bytes(int fm) { return (size_t)SCAN_WARPS * CQ_CAP * 8 + (size_t)SCAN_WARPS * hl_cap(fm) * 2; }
constexpr size_t SCAN_SMEM_BYTES = (size_t)BLOOM_WORDS * 4 + scan_lists_bytes(0);
// L2 filter mode keeps only the lists in shared memory: the rest of the 256 KB stays L1, whose
// lines are what outstanding global loads are tracked in (a 30 KB L1 caps an SM at ~0.3
// random loads per clock against 1.0 with a large one: scripts/micro/l2_gather.cu).
constexpr size_t SCAN_SMEM_BYTES_GF = scan_lists_bytes(1);       // L2 filter, no pre-filter
constexpr size_t SCAN_SMEM_BYTES_PRE = scan_lists_bytes(2);      // + pre_words * 4
constexpr int MACRO_GS = 2;  // sub-tiles per group of the macro path

constexpr int MAX_SEED_LEN = 15;             // 30 bits: leaves SEED_EMPTY outside the seed space
constexpr uint32_t SEED_MULT = 0x9E3779B1u;  // odd multiplier of the filter hash
constexpr uint32_t PRE_REHASH = 0x85EBCA6Bu;  // odd: L2-filter hash behind a pre-filter = h * PRE_REHASH
constexpr uint32_t SEEDTAB_MULT = 0xC2B2AE3Du; // seed slot = mulhi(seed * SEEDTAB_MULT, n_slots)
constexpr uint32_t SEED_EMPTY = 0xFFFFFFFFu;  // free slot of the sizing set (k_assign_seeds, count_only)
// Seed-table slot word: bits 0..29 the seed, bit 30 = slot is free, bit 31 = some seed
// whose home is this slot lives further along (a miss must walk on).  A free slot is the
// memset pattern 0x40.
constexpr uint32_t ST_EMPTY = 0x40404040u;
constexpr uint32_t ST_FREE_BIT = 0x40000000u;
constexpr uint32_t ST_MOVED_BIT = 0x80000000u;
constexpr uint32_t ST_SEED_BITS = 0x7FFFFFFFu;  // (word & ST_SEED_BITS) == seed  <=>  the slot holds it
constexpr uint64_t KEY_EMPTY = ~0ull;        // keys use at most 62 bits
constexpr uint32_t ENTRY_DEAD = 0xFFFFFFFFu; // repeated (key, owner) triple
constexpr int KBUCKET = 2;                   // slots per key-table bucket (32 B, one L2 sector)

// ---- hashes ----------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t hash32(uint32_t x) {
  x *= 0x85EBCA6Bu;
  x ^= x >> 15;
  x *= 0xC2B2AE35u;
  x ^= x >> 16;
  return x;
}

// home slot of a seed in the exact seed table: multiplicative hash, range-reduced by a
// multiply-high so that the table need not be a power of two (a table rounded up to one was
// up to twice the size it had to be, all of it L2 footprint)
__host__ __device__ __forceinline__ uint32_t seed_home(uint32_t seed, uint32_t n_slots) {
  return (uint32_t)(((uint64_t)(seed * SEEDTAB_MULT) * n_slots) >> 32);
}

// Seed filter: a blocked Bloom filter, all bits of a seed inside one 32-bit word.  With
// h = seed * seed_mult and the 64-bit product h * n_words: the word is the product's high
// half, bit 1 is (seed & 31), bits 2..4 are 5-bit fields taken from the top of the
// product's LOW half - so one IMAD.WIDE yields the word and every hashed bit index.  (A
// multiply-high per index costs 5 issue cycles per warp on sm_100 and stalls the ALU pipe
// meanwhile, against 2.4 for IMAD.WIDE: scripts/micro/int_pipes.cu.)
__host__ __device__ __forceinline__ uint32_t bloom_word(uint32_t h, uint32_t n_words) {
  return (uint32_t)(((uint64_t)h * n_words) >> 32);
}
__host__ __device__ __forceinline__ uint32_t bloom_bits(uint32_t seed, uint32_t h, uint32_t n_words,
                                                        int n_hashes) {
  const uint32_t lo = (uint32_t)((uint64_t)h * n_words);
  uint32_t bits = 1u << (seed & 31);
  if (n_hashes >= 2) bits |= 1u << (lo >> 27);
  if (n_hashes >= 3) bits |= 1u << ((lo >> 22) & 31);
  if (n_hashes >= 4) bits |= 1u << ((lo >> 17) & 31);
  return bits;
}

__host__ __device__ __forceinline__ uint64_t kmer_mask(int k) { return (1ull << (2 * k)) - 1; }

// The L2 filter modes key their seeds by the strand-canonical form of the s-mer, min(s-mer,
// its reverse complement).  Both orientations of a haplotype then share their seeds: half the
// seeds in the filters and the seed table, for ~7 more instructions per lookup.
__host__ __device__ constexpr bool canon_for_mode(int fm) { return fm > 0; }

// Reverse complement of an s-mer held in the low 2s bits (stream order either way: first base
// least significant), cshift = 32 - 2s; x must be masked to its 2s bits.
__device__ __forceinline__ uint32_t seed_revcomp(uint32_t x, uint32_t cshift) {
  const uint32_t r = __brev(x);  // bases reversed (now in the top 2s bits), the two bits of each base swapped
  // swap them back and complement in ONE LOP3: ~(((r >> 1) & 0x55555555) | ((r << 1) & ~0x55555555))
  uint32_t c;
  asm("lop3.b32 %0, %1, %2, 0x55555555, 0x1B;" : "=r"(c) : "r"(r >> 1), "r"(r << 1));
  return c >> cshift;      // realign (the ones below the s-mer are shifted out)
}
// Canonical seed and whether the s-mer had to be flipped to get it.
__device__ __forceinline__ uint32_t seed_canon(uint32_t x, uint32_t cshift, uint32_t &flip) {
  const uint32_t r = seed_revcomp(x, cshift);
  flip = r < x;
  return r < x ? r : x;
}

// Reverse the order of the k bases of a 2k-bit value (an involution).  Turns
// a key (first base most significant) into stream order (first base least
// significant) and back.
__device__ __forceinline__ uint64_t base_reverse(uint64_t v, int k) {
  uint64_t r = __brevll(v);
  r = ((r >> 1) & 0x5555555555555555ull) | ((r & 0x5555555555555555ull) << 1);
  return r >> (64 - 2 * k);
}

// ---- L2 residency hints ------------------------------------------------------------
// The stream is read once (evict-first); the seed / key tables and the counters
// are re-read for the whole launch and should stay in the 126 MB L2 (evict-last).
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint4 ldg_v4_hint(const void *ptr, uint64_t pol) {
  uint4 v;
  asm volatile("ld.global.nc.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(ptr), "l"(pol));
  return v;
}
__device__ __forceinline__ uint32_t ldg_u32_hint(const void *ptr, uint64_t pol) {
  uint32_t v;
  asm volatile("ld.global.nc.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(ptr), "l"(pol));
  return v;
}
__device__ __forceinline__ uint64_t ldg_u64_hint(const void *ptr, uint64_t pol) {
  uint64_t v;
  asm volatile("ld.global.nc.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(v) : "l"(ptr), "l"(pol));
  return v;
}

// ---- the two lookup structures (both in L2) -----------------------------------
// Seed table: open addressing, linear probing, 64-byte slots of two 32-byte HALVES (one L2
// sector each).  A half holds the seed AND a record, so a verified seed costs no further
// dependent load.  Half 0 is the record for reads that show the seed as stored; half 1 (used
// only with canonical seeds) the record for reads that show its reverse complement - each is
// written in the orientation of the reads that will be compared with it.  Words of a half:
//   word 0   (half 0 only) bits 0..29 the seed, bit 30 = slot is free, bit 31 = some seed whose
//            home is this slot lives further along (a miss must walk on); see ST_*
//   word 1   info: bit j = some key designates this seed at offset j (its window starts j
//            bases before the seed); bit 31 (INFO_DIRECT) = a DIRECT record, below
//   word 2-4 nb, the NEIGHBOURHOOD: the 48 bases from E = k - s before the seed, 2 bits each,
//            stream order - the union of all windows that designate the seed (2k - s <= 48)
//   word 5-7 wild: both bits of a base set where the designating keys disagree, or none covers it
// A DIRECT record (the build proves it, DESIGN.md §4) has every designation from one variant, at
// most one per (offset j, allele), entry = c_a + sigma_a * j within allele a, and its windows agree
// on every covered base except at most one, X (an SNV's base), which each allele shows one way.
// Its wild mask is "not covered, or X": the covered range follows from info's lowest and highest
// offset, so words 5-7 carry instead
//   word 5, 6  c_0, c_1
//   word 7     bits 0..5 X; bits 6..9: read bases at X that pick allele 0 (bit 6 + base);
//              bits 10..13: those that pick allele 1; bit 14 / 15: sigma_0 / sigma_1 = -1
// (a record that only one allele designates has no X: that allele takes every base at X = E, the
// seed's first base, which the read matches anyway).  Stage C counts its windows straight from
// the record, without the key table.
// A lookup is ONE 4-byte load of word 0 unless the home slot carries ST_MOVED_BIT: a seed
// absent from an unmarked home slot is absent from the table.
// A read window can equal a designating key only if the read equals nb on the window's
// bases outside wild.  Stage C therefore compares the read with nb once and probes the key
// table only for windows inside the matching run around the seed: an s-mer that equals a
// seed by chance (1 lookup in 1300 at s = 14 with 200 k seeds) costs a compare instead of
// ~16 dependent key-table probes that miss L2.
// Shared-memory filter mode only: filter false positives are frequent there, and at the
// slot table's load factor (1/2) a third of them would land on a slot that says "walk on".
// A PROBE ARRAY in front takes them: one 4-byte word per entry (same ST_* encoding), 1/8 full,
// so that an absent seed costs one 4-byte load (about one in a hundred a second one); only
// seeds found in it go on to their slot.  n_probe = 0: no probe array (L2 filter modes,
// where false positives are rare and true seeds would only pay an extra hop).
struct SeedTable {
  uint4 *slots;      // 4 x uint4 per slot (2 per half)
  uint32_t n_slots;  // any size (not a power of two)
  uint32_t *probe;
  uint32_t n_probe;
};
__host__ __device__ __forceinline__ uint32_t seed_next(uint32_t slot, uint32_t n_slots) {
  return slot + 1 == n_slots ? 0u : slot + 1;
}
constexpr int NB_BASES = 48;
constexpr uint32_t INFO_DIRECT = 0x80000000u;  // info bit of a direct record (offsets j <= k - s <= 23)
constexpr uint32_t INFO_OFFSETS = 0x00FFFFFFu;
constexpr int DIR_PICK0 = 6, DIR_PICK1 = 10, DIR_NEG0 = 14, DIR_NEG1 = 15;  // word 7 of a direct record
// Key table: 16-byte slots {key lo, key hi, entry index, packed designated
// offsets}, buckets of 2 slots = one 32-byte L2 sector (two LDG.128), a
// multimap: one slot per (key, owner) entry; a full bucket spills into the next.
// Packed offsets: field f = orientation * D + class, 32 / (2 D) bits wide, holds
// j / D of the designated seed offset j = (j / D) * D + class.
struct KeyTable {
  uint4 *slots;
  uint32_t bucket_mask;  // n_buckets - 1
};
// Keys are genome k-mers (already well spread): a 32-bit fold-multiply is enough and
// costs a fifth of a 64-bit finaliser in stage C.
__host__ __device__ __forceinline__ uint32_t key_bucket(uint64_t key, uint32_t bucket_mask) {
  uint32_t x = (uint32_t)key ^ ((uint32_t)(key >> 32) * 0x9E3779B1u);
  x *= 0x85EBCA6Bu;
  x ^= x >> 15;
  return x & bucket_mask;
}
__host__ __device__ __forceinline__ uint64_t slot_key(const uint4 &s) {
  return (uint64_t)s.y << 32 | s.x;
}
// designated offset stored in a slot for (orientation, class)
__host__ __device__ __forceinline__ uint32_t slot_offset(uint32_t packed, int ori, int cls, int D) {
  const int W = 32 / (2 * D);
  return ((packed >> (W * (ori * D + cls))) & ((1u << W) - 1)) * D + cls;
}

// ---- parameters of one scan launch -------------------------------------------
// A launch scans up to MAX_SEGMENTS packed streams (e.g. the three samples of a trio) one
// after the other in one grid: work units are numbered across the segments.
constexpr int MAX_SEGMENTS = 4;
struct ScanSegment {
  const uint32_t *bases;  // 2-bit stream, 16 positions per word
  const uint32_t *mask;   // 1-bit validity stream, 32 positions per word
  uint32_t *counts;       // the sample's [n_entries] counters
  uint32_t n_pos, n_bwords, n_mwords, n_tiles;
  uint32_t unit_begin;    // first work unit (tile, or macro tile) of this segment
  uint32_t unit_end;      // first work unit AFTER this segment
};
struct ScanParams {
  ScanSegment seg[MAX_SEGMENTS];
  int n_seg;
  const uint32_t *bloom;  // seed filter: BLOOM_WORDS words copied into shared memory per CTA,
                          // or (large candidate sets) bloom_words words probed in L2
  uint32_t bloom_words;
  // L2 filter mode only: optional one-bit pre-filter in shared memory (pre_words words, 0 =
  // none); only its hits go on to the L2 filter, which is then hashed with h * PRE_REHASH.
  const uint32_t *pre;
  uint32_t pre_words;
  SeedTable st;
  KeyTable kt;
  uint32_t seed_mult;  // SEED_MULT << (32 - 2s): the product ignores bases beyond s
  uint32_t seed_mask;  // low 2s bits
  uint32_t cshift;     // 32 - 2s (seed_revcomp)
  uint32_t four;       // = 4, opaque to the compiler: keeps the filter address on the FMA pipe
  uint32_t pw[32];     // pw[n] = 2^n, opaque too: multiplies by these stay on the FMA pipe
  uint32_t filter_words;  // = BLOOM_WORDS (shared-memory mode), as a run-time operand of the wide multiply
  int k, s;
  unsigned long long *prof;  // 4 counters or nullptr
  // ---- region mode only (k_scan<..., RG = true>).  Kept at the end so that the whole-stream
  // kernels' parameter offsets stay where they were.  The read-locus index of every segment of
  // the launch is one set of concatenated arrays: reads are numbered across the segments.
  const uint32_t *read_start;   // [n_reads] first stream position of read r, inside its segment
  const uint32_t *tile_read;    // per segment, at rseg[i].tile_base: [n_tiles + 1] the first read
                                // reaching into 2048-position tile t; the last entry is the
                                // segment's last read
  const ulonglong2 *read_span;  // [n_reads] the read's alignment interval {lo, hi}; {*, 0} if empty
  const ulonglong2 *entry_win;  // [n_entries] the window of the entry's variant; {*, 0} if empty
  struct {
    uint32_t tile_base;  // first entry of the segment's hints in tile_read
    uint32_t n_tiles;    // its 2048-position tiles
  } rseg[MAX_SEGMENTS];
};

// Region mode: positions per tile of the read-locus index (a position resolves to its read with
// one hint load and a binary search between two neighbouring hints).
constexpr int LOCI_TILE_SHIFT = 11;

// Half-open intervals overlap.  Both are normalised so that an empty one has hi = 0, which no
// unsigned lo is below: an empty read or window never overlaps anything.
__host__ __device__ __forceinline__ bool spans_overlap(ulonglong2 a, ulonglong2 b) {
  return a.x < b.y && b.x < a.y;
}

}  // namespace dkb

// dkb_build.cuh — kernel 1 (table build) and kernel 3 (finalise).
//
// Build = the GPU form of src/counter.rs's "set of k-mers that span each
// candidate allele" (unmounted; DESIGN.md §2): every entry (canonical key,
// variant, allele) gets a slot in a bucketised open-addressing multimap; for
// both orientations of the key and every stride class one s-mer of the k-mer
// is designated as its seed and put in the exact seed table and the filter.
#pragma once
#include "../../include/dkb.h"
#include "dkb_device.cuh"

namespace dkb {

struct BuildParams {
  const uint64_t *keys;
  const uint32_t *variant;
  const uint8_t *allele;
  const uint16_t *win_index;  // may be null: bit 15 = haplotype window is the rc of the key
  const uint16_t *win_count;  // may be null
  uint32_t n;
  KeyTable kt;
  uint32_t *slot_of;  // [n] slot claimed by each entry
  uint8_t *dead;      // [n]
  int k, s, D;
  int canon;  // seeds are keyed by min(s-mer, its reverse complement)
};

// Claim one free slot for every entry: home bucket first, then the following
// buckets.  A multimap: equal keys take separate slots.
__global__ void k_insert_entries(const BuildParams B) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B.n) return;
  const uint64_t key = B.keys[i];
  uint32_t b = key_bucket(key, B.kt.bucket_mask);
  while (true) {
    for (int j = 0; j < KBUCKET; j++) {
      const uint32_t slot = b * KBUCKET + j;
      if (atomicCAS(reinterpret_cast<unsigned long long *>(B.kt.slots + slot), KEY_EMPTY, key) ==
          KEY_EMPTY) {
        B.kt.slots[slot].z = i;
        B.kt.slots[slot].w = 0;  // packed offsets, OR-ed in by k_assign_seeds
        B.slot_of[i] = slot;
        return;
      }
    }
    b = (b + 1) & B.kt.bucket_mask;
  }
}

// An entry is dead when an earlier entry has the same (key, variant, allele).
__global__ void k_mark_repeats(const BuildParams B) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B.n) return;
  const uint64_t key = B.keys[i];
  uint32_t b = key_bucket(key, B.kt.bucket_mask);
  uint8_t dead = 0;
  bool open = false;
  while (!open && !dead) {
    for (int j = 0; j < KBUCKET; j++) {
      const uint4 sl = B.kt.slots[b * KBUCKET + j];
      const uint64_t tk = slot_key(sl);
      if (tk == KEY_EMPTY) {
        open = true;
      } else if (tk == key) {
        const uint32_t e = sl.z;
        if (e < i && B.variant[e] == B.variant[i] && B.allele[e] == B.allele[i]) dead = 1;
      }
    }
    b = (b + 1) & B.kt.bucket_mask;
  }
  B.dead[i] = dead;
}

__global__ void k_apply_dead(const BuildParams B) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B.n) return;
  if (B.dead[i]) B.kt.slots[B.slot_of[i]].z = ENTRY_DEAD;
}

// Word w of half h (0, 1) of seed-table slot `slot` (layout in dkb_device.cuh).
__device__ __forceinline__ uint32_t *slot_word(const SeedTable &T, uint32_t slot, int w, int h = 0) {
  return reinterpret_cast<uint32_t *>(T.slots) + 16 * (size_t)slot + 8 * h + w;
}

// Insert a seed into the seed table: the home slot, else the first free slot after it,
// with the home slot marked ST_MOVED_BIT so that lookups know to walk on.
__device__ __forceinline__ void seedtab_insert(const SeedTable &T, uint32_t seed) {
  uint32_t slot = seed_home(seed, T.n_slots);
  bool home = true;
  while (true) {
    uint32_t *w0 = slot_word(T, slot, 0);
    uint32_t old = *reinterpret_cast<volatile uint32_t *>(w0);
    if (old & ST_FREE_BIT) {
      old = atomicCAS(w0, ST_EMPTY, seed);
      if (old == ST_EMPTY) old = seed;
    }
    if ((old & ST_SEED_BITS) == seed) return;
    if (home) atomicOr(w0, ST_MOVED_BIT);  // taken by another seed
    home = false;
    slot = seed_next(slot, T.n_slots);
  }
}

// Same insertion into the probe array (one word per entry).
__device__ __forceinline__ void probe_insert(const SeedTable &T, uint32_t seed) {
  uint32_t e = seed_home(seed, T.n_probe);
  bool home = true;
  while (true) {
    uint32_t old = *reinterpret_cast<volatile uint32_t *>(T.probe + e);
    if (old & ST_FREE_BIT) {
      old = atomicCAS(T.probe + e, ST_EMPTY, seed);
      if (old == ST_EMPTY) old = seed;
    }
    if ((old & ST_SEED_BITS) == seed) return;
    if (home) atomicOr(T.probe + e, ST_MOVED_BIT);
    home = false;
    e = seed_next(e, T.n_probe);
  }
}

// Slot of a seed that is in the table.
__device__ __forceinline__ uint32_t seedtab_find(const SeedTable &T, uint32_t seed) {
  uint32_t slot = seed_home(seed, T.n_slots);
  while ((*slot_word(T, slot, 0) & ST_SEED_BITS) != seed) slot = seed_next(slot, T.n_slots);
  return slot;
}

// Working form of a slot's record while the designations are being collected (words 1..7):
// {info, OR of the windows' bases [3], AND of (bases | not covered) [3]}; cov[3] per slot =
// union of the windows' extents.  k_finish_records turns it into the final form.
__device__ __forceinline__ void record_add(uint32_t *rec, uint32_t *cov, int j, uint64_t v, int k,
                                           int E) {
  atomicOr(rec + 1, 1u << j);
  if (E + k > NB_BASES) return;  // neighbourhood does not fit: records stay all-wild
  const int o = E - j;           // first base of the window inside the neighbourhood
  const unsigned __int128 val = (unsigned __int128)v << (2 * o);
  const unsigned __int128 ext = (unsigned __int128)kmer_mask(k) << (2 * o);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const uint32_t vw = (uint32_t)(val >> (32 * i)), ew = (uint32_t)(ext >> (32 * i));
    if (ew == 0) continue;
    atomicOr(rec + 2 + i, vw);
    atomicAnd(rec + 5 + i, vw | ~ew);
    atomicOr(cov + i, ew);
  }
}

// Every slot free, both its records in the (empty) working form.
__global__ void k_init_slots(const SeedTable T) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per uint4
  if (i >= 4 * (size_t)T.n_slots) return;
  T.slots[i] = (i & 1) ? make_uint4(0u, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu)
                       : make_uint4(ST_EMPTY, 0u, 0u, 0u);
}

__global__ void k_finish_records(const SeedTable T, const uint32_t *cov) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per half
  if (i >= 2 * (size_t)T.n_slots) return;
  if (*slot_word(T, (uint32_t)(i >> 1), 0) & ST_FREE_BIT) return;
  uint32_t *r = slot_word(T, (uint32_t)(i >> 1), 0, (int)(i & 1));
#pragma unroll
  for (int w = 0; w < 3; w++) {
    const uint32_t d = r[2 + w] ^ r[5 + w];               // bases on which the windows disagree
    const uint32_t t = (d | d >> 1) & 0x55555555u;
    r[5 + w] = ~cov[(size_t)i * 3 + w] | t | t << 1;      // wild: not covered, or disagreement
  }
}

// ---- direct records (dkb_device.cuh; the proof is in DESIGN.md §4) ----------------------
// Build scratch per record half, 8 words, zeroed: what its designations have in common.
//   0     variant + 1                  1, 2  allele 0: e - j + 32, e + j + 1 (entry e, offset j)
//   3, 4  the same for allele 1        5, 6  A0, A1: offsets designated by allele 0, 1
//   7     flags: bit 4a + b = a window of allele a shows base b at X; DIRF_* below
// Words 0-4 keep the first value written; a later designation with another value sets a flag.
constexpr int DIR_WORDS = 8;
constexpr uint32_t DIRF_REJECT = 1u << 8;    // a key with a second live owner, or a window without X
constexpr uint32_t DIRF_VARIANT = 1u << 9;   // more than one variant
constexpr uint32_t DIRF_SLOPE = 1u << 10;    // << 2a: e - j varies in allele a; << 2a + 1: e + j varies

__device__ __forceinline__ void dir_same(uint32_t *w, uint32_t v, uint32_t *flags, uint32_t bit) {
  const uint32_t old = atomicCAS(w, 0u, v);
  if (old != 0u && old != v) atomicOr(flags, bit);
}

// Bases of a finished record (words 5-7 = wild) that are wild inside the covered range, i.e.
// disputed by the designating windows: their number, and x = the first of them.
__device__ __forceinline__ int disputed_bases(const uint32_t *rec, const uint32_t *cov, int &x) {
  int n = 0;
  x = 0;
  for (int w = 2; w >= 0; w--) {
    const uint32_t d = rec[5 + w] & cov[w];
    n += __popc(d);
    if (d) x = 16 * w + ((__ffs(d) - 1) >> 1);
  }
  return n >> 1;
}

// One designation (entry e of variant `var`, allele a, offset j, window v in stream order) into
// the scratch d of its record half; `shared` = another live entry has e's key.
__device__ __forceinline__ void direct_add(const uint32_t *rec, const uint32_t *cov, uint32_t *d,
                                           uint32_t e, uint32_t var, int a, int j, uint64_t v, int k,
                                           int E, bool shared) {
  uint32_t *const flags = d + 7;
  if (shared) atomicOr(flags, DIRF_REJECT);
  atomicOr(d + 5 + a, 1u << j);
  dir_same(d, var + 1, flags, DIRF_VARIANT);
  dir_same(d + 1 + 2 * a, e - j + 32, flags, DIRF_SLOPE << (2 * a));
  dir_same(d + 2 + 2 * a, e + j + 1, flags, DIRF_SLOPE << (2 * a + 1));
  if (E + k > NB_BASES) return;  // no neighbourhood: never direct
  int x;
  if (disputed_bases(rec, cov, x) != 1) return;  // none, or too many (k_finish_direct decides)
  const int o = E - j;                            // first base of the window in the neighbourhood
  if (x < o || x >= o + k) atomicOr(flags, DIRF_REJECT);
  else atomicOr(flags, 1u << (4 * a + (uint32_t)((v >> (2 * (x - o))) & 3)));
}

// One thread per record half: make the half direct where its designations allow it.
// stats[0] += occupied halves, stats[1] += direct ones.
__global__ void k_finish_direct(const SeedTable T, const uint32_t *cov, const uint32_t *dir, int k,
                                int s, unsigned long long *stats) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per half
  const int E = k - s;
  bool occ = false, direct = false;
  if (i < 2 * (size_t)T.n_slots && !(*slot_word(T, (uint32_t)(i >> 1), 0) & ST_FREE_BIT)) {
    uint32_t *r = slot_word(T, (uint32_t)(i >> 1), 0, (int)(i & 1));
    occ = r[1] != 0;
    const uint32_t *d = dir + i * DIR_WORDS;
    const uint32_t A0 = d[5], A1 = d[6], f = d[7];
    const uint32_t seen0 = f & 0xFu, seen1 = (f >> 4) & 0xFu;
    int x;
    const int nx = disputed_bases(r, cov + i * 3, x);
    direct = occ && E + k <= NB_BASES && !(f & (DIRF_REJECT | DIRF_VARIANT));
    uint32_t pick0 = 0xFu, pick1 = 0xFu;
    if (A0 && A1) {  // an SNV's two alleles: the same offsets, and one disputed base each shows its own way
      direct = direct && A0 == A1 && nx == 1 && __popc(seen0) == 1 && __popc(seen1) == 1 && seen0 != seen1;
      pick0 = seen0;
      pick1 = seen1;
    } else {  // one allele: no disputed base; X = the seed's first base, which every read matches
      direct = direct && nx == 0;
      x = E;
      if (!A0) pick0 = 0;
      if (!A1) pick1 = 0;
    }
    uint32_t c[2] = {0, 0}, neg = 0;
    for (int a = 0; a < 2; a++) {
      if (!(a ? A1 : A0)) continue;
      if (!(f & (DIRF_SLOPE << (2 * a)))) {
        c[a] = d[1 + 2 * a] - 32;  // e = c + j
      } else if (!(f & (DIRF_SLOPE << (2 * a + 1)))) {
        c[a] = d[2 + 2 * a] - 1;   // e = c - j
        neg |= 1u << a;
      } else {
        direct = false;
      }
    }
    if (direct) {
      r[5] = c[0];
      r[6] = c[1];
      r[7] = (uint32_t)x | pick0 << DIR_PICK0 | pick1 << DIR_PICK1 | (neg & 1u) << DIR_NEG0 |
             (neg >> 1) << DIR_NEG1;
      r[1] |= INFO_DIRECT;
    }
  }
  const uint32_t n_occ = __popc(__ballot_sync(FULL_MASK, occ)), n_dir = __popc(__ballot_sync(FULL_MASK, direct));
  if ((threadIdx.x & 31) == 0) {
    if (n_occ) atomicAdd(stats, (unsigned long long)n_occ);
    if (n_dir) atomicAdd(stats + 1, (unsigned long long)n_dir);
  }
}

// popcount of n words / number of zero bytes, for the build statistics (out[0], out[1])
__global__ void k_build_stats(const uint32_t *words, uint32_t n_words, const uint8_t *dead,
                              uint32_t n_dead, unsigned long long *out) {
  unsigned long long bits = 0, live = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_words;
       i += (size_t)gridDim.x * blockDim.x)
    bits += __popc(words[i]);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_dead;
       i += (size_t)gridDim.x * blockDim.x)
    live += dead[i] == 0;
  for (int o = 16; o; o >>= 1) {
    bits += __shfl_xor_sync(FULL_MASK, bits, o);
    live += __shfl_xor_sync(FULL_MASK, live, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (bits) atomicAdd(out, bits);
    if (live) atomicAdd(out + 1, live);
  }
}

// Count distinct seeds with a plain open-addressing set (sizing pass).
__device__ __forceinline__ void seedset_insert(uint32_t *set, uint32_t mask, uint32_t seed,
                                               unsigned int *n_new) {
  uint32_t slot = hash32(seed) & mask;
  while (true) {
    uint32_t old = set[slot];
    if (old == SEED_EMPTY) old = atomicCAS(set + slot, SEED_EMPTY, seed);
    if (old == SEED_EMPTY) {
      atomicAdd(n_new, 1u);
      return;
    }
    if (old == seed) return;
    slot = (slot + 1) & mask;
  }
}

// One thread per (entry, orientation): choose the designated seed offset of
// every stride class.
//   ladder rule (window hints present): seeds sit on a ladder of spacing
//     G = floor((k-s+1)/D)*D along the haplotype, so neighbouring windows share
//     them (2 seeds per SNV haplotype strand and class at k=31, s<=15);
//   min-hash rule (no hints): the s-mer of the class with the smallest hash.
// Four passes (the choice of offsets is the same in each):
//   ASSIGN_COUNT   add the seeds to `set` (sizing);
//   ASSIGN_INSERT  record the offsets in the entry's slot, insert the seeds, set their filter bits;
//   ASSIGN_RECORD  add offset and window to the record in the seed's slot;
//   ASSIGN_DIRECT  (after k_finish_records) add the designation to the direct-record scratch `dir`.
enum { ASSIGN_COUNT = 0, ASSIGN_INSERT = 1, ASSIGN_RECORD = 2, ASSIGN_DIRECT = 3 };
__global__ void k_assign_seeds(const BuildParams B, int pass, uint32_t *set, uint32_t set_mask,
                               unsigned int *n_seeds, const SeedTable T, uint32_t *cov,
                               uint32_t *bloom, uint32_t bloom_words, uint32_t *pre,
                               uint32_t pre_words, uint32_t seed_mult, int n_hashes, uint32_t *dir) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t i = t >> 1;
  const int ori = t & 1;
  if (i >= B.n || B.dead[i]) return;
  const int k = B.k, s = B.s, D = B.D, E = k - s;
  const uint64_t km = kmer_mask(k);
  const uint64_t key = B.keys[i];
  const uint64_t v0 = base_reverse(key, k);  // stream order of the key's own string
  const uint64_t v1 = ~key & km;             // stream order of its reverse complement
  if (ori == 1 && v1 == v0) return;          // palindrome: one orientation only
  const uint64_t v = ori ? v1 : v0;
  const uint32_t smask = (1u << (2 * s)) - 1;
  const bool ladder = B.win_index != nullptr && B.win_count != nullptr;
  uint32_t u = 0;
  if (ladder) {
    const uint32_t wi = B.win_index[i];
    const uint32_t nwin = B.win_count[i];
    const int hap_ori = (wi >> 15) & 1;  // orientation whose string reads along the haplotype
    u = wi & 0x7FFFu;
    if (ori != hap_ori) u = nwin - 1 - u;  // same window seen on the other strand
  }
  bool shared = false;  // ASSIGN_DIRECT: another live entry has this key (k_mark_repeats' walk)
  if (pass == ASSIGN_DIRECT) {
    uint32_t b = key_bucket(key, B.kt.bucket_mask);
    for (bool open = false; !open && !shared; b = (b + 1) & B.kt.bucket_mask) {
      for (int q = 0; q < KBUCKET; q++) {
        const uint4 sl = B.kt.slots[b * KBUCKET + q];
        const uint64_t tk = slot_key(sl);
        if (tk == KEY_EMPTY) open = true;
        else if (tk == key && sl.z != ENTRY_DEAD && sl.z != i) shared = true;
      }
    }
  }
  uint32_t offs = 0;
  const int W = 32 / (2 * D);  // bits per packed offset field
  for (int c = 0; c < D; c++) {
    int j;
    if (ladder) {
      const int G = ((E + 1) / D) * D;
      const int r = (int)((u + c) % D);
      const int base = E - ((E - r) % D);  // largest ladder origin <= E in residue r
      int P = base;
      if ((int)u > base) P = base + (((int)u - base + G - 1) / G) * G;
      j = P - (int)u;
    } else {
      uint32_t best = 0xFFFFFFFFu;
      j = c;
      for (int o = c; o <= E; o += D) {
        const uint32_t sc = hash32((uint32_t)(v >> (2 * o)) & smask);
        if (sc < best) {
          best = sc;
          j = o;
        }
      }
    }
    uint32_t seed = (uint32_t)(v >> (2 * j)) & smask, flip = 0;
    // canonical seeds: the seed is stored once for both strands; reads that show this
    // orientation of it are served by half `flip` of its slot
    if (B.canon) seed = seed_canon(seed, 32 - 2 * s, flip);
    if (pass == ASSIGN_COUNT) {
      seedset_insert(set, set_mask, seed, n_seeds);
    } else if (pass == ASSIGN_INSERT) {
      offs |= (uint32_t)(j / D) << (W * (ori * D + c));
      seedtab_insert(T, seed);
      if (T.n_probe) probe_insert(T, seed);
      uint32_t h = seed * seed_mult;
      if (pre_words) {  // one-bit pre-filter; the main filter behind it uses an independent hash
        atomicOr(pre + bloom_word(h, pre_words), 1u << ((uint32_t)((uint64_t)h * pre_words) >> 27));
        h *= PRE_REHASH;
      }
      atomicOr(bloom + bloom_word(h, bloom_words), bloom_bits(seed, h, bloom_words, n_hashes));
    } else {
      const uint32_t slot = seedtab_find(T, seed);
      const size_t h = (size_t)slot * 2 + flip;
      if (pass == ASSIGN_RECORD)
        record_add(slot_word(T, slot, 0, (int)flip), cov + h * 3, j, v, k, E);
      else
        direct_add(slot_word(T, slot, 0, (int)flip), cov + h * 3, dir + h * DIR_WORDS, i, B.variant[i],
                   B.allele[i], j, v, k, E, shared);
    }
  }
  if (pass == ASSIGN_INSERT) atomicOr(&B.kt.slots[B.slot_of[i]].w, offs);
}

// ---- kernel 3: finalise -----------------------------------------------------
// NS samples (3: a trio; 2 + n_children in a family).
// counts: [NS][n]; hits/distinct: [n_variants][2][NS]; n_kmers: [n_variants][2]
// A (variant, allele, sample) hit total saturates at UINT32_MAX instead of wrapping: the sum of
// up to 32 u32 counters is formed from their 16-bit halves in 64 bits, and a leader whose
// atomicAdd wrapped the cell sets it to UINT32_MAX.  Until the first wrap the cell holds the exact
// partial sum; after it, every add wraps again (the cell is UINT32_MAX or wrapped), so the last
// operation on the cell is an exchange: the cell ends at UINT32_MAX exactly when the total passes
// it.  The NS adds are issued back to back and checked after (one round trip per leader).  The
// calls of k_calls then equal the rule on the exact sums for every max_parent_alt_hits below
// UINT32_MAX.
template <int NS>
__global__ void k_variant_reduce(const uint32_t *counts, const uint32_t *variant,
                                 const uint8_t *allele, const uint8_t *dead, uint32_t n,
                                 uint32_t *hits, uint32_t *distinct, uint32_t *n_kmers) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = i < n && !dead[i];
  // Entries of one (variant, allele) usually sit next to each other (the host builder emits
  // them so): the lanes of a warp that share an owner add up among themselves (REDUX) and one
  // of them issues the atomics - ~10x fewer than one set per entry.  Any order stays correct.
  const uint32_t va = live ? variant[i] * 2u + allele[i] : 0xFFFFFFFFu;
  uint32_t c[NS] = {};
  if (live) {
#pragma unroll
    for (int smp = 0; smp < NS; smp++) c[smp] = counts[(size_t)smp * n + i];
  }
  const unsigned peers = __match_any_sync(FULL_MASK, va);
  const bool leader = live && (__ffs(peers) - 1) == (int)(threadIdx.x & 31);
  const uint32_t nk = __reduce_add_sync(peers, live ? 1u : 0u);
  uint32_t h[NS], d[NS];
#pragma unroll
  for (int smp = 0; smp < NS; smp++) {
    const uint64_t sum = ((uint64_t)__reduce_add_sync(peers, c[smp] >> 16) << 16) +
                         __reduce_add_sync(peers, c[smp] & 0xFFFFu);
    h[smp] = sum > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)sum;
    d[smp] = __reduce_add_sync(peers, c[smp] ? 1u : 0u);
  }
  if (!leader) return;
  atomicAdd(n_kmers + va, nk);
#pragma unroll
  for (int smp = 0; smp < NS; smp++) {
    if (h[smp]) {
      c[smp] = atomicAdd(hits + (size_t)va * NS + smp, h[smp]);  // c: the cell before the add
      atomicAdd(distinct + (size_t)va * NS + smp, d[smp]);
    }
  }
#pragma unroll
  for (int smp = 0; smp < NS; smp++)
    if (h[smp] && c[smp] + h[smp] < c[smp]) atomicExch(hits + (size_t)va * NS + smp, 0xFFFFFFFFu);
}

struct Thresholds {
  uint32_t min_child_alt_hits, min_child_alt_distinct, max_parent_alt_hits, min_parent_ref_hits;
};

// Child sexes of one kernel 3 (DKB_SEX_*), by value: child c's in bits 2c, 2c + 1 (at most
// DKB_MAX_CHILDREN of them; a word instead of an array, which indexing would put on the stack).
typedef uint32_t ChildSexes;

// Which parents' clauses apply to a child of sex `sex` at a locus of class `cls` (DESIGN.md §2
// "Inheritance"): bit 0 the mother's, bit 1 the father's; bit 2 = the child has no copy of the
// locus (a daughter at Y), which the call reports as DKB_CALL_NO_COPY.
__device__ __forceinline__ uint32_t parent_clauses(uint32_t cls, uint32_t sex) {
  switch (cls) {
    case DKB_LOCUS_X: return sex == DKB_SEX_MALE ? 1u : 3u;
    case DKB_LOCUS_Y: return sex == DKB_SEX_MALE ? 2u : sex == DKB_SEX_FEMALE ? 4u : 3u;
    case DKB_LOCUS_MATERNAL: return 1u;
    default: return 3u;
  }
}

// One thread per (variant, child): the trio rule on child ch's alt support and the hits of the
// parents whose clauses apply at variant v's locus class (cls[v], all autosomal when cls is
// null) for child ch's sex; calls: [n_variants][NS - 2].  n_items = n_variants * (NS - 2).
template <int NS>
__global__ void k_calls(const uint32_t *hits, const uint32_t *distinct, uint32_t n_items,
                        const Thresholds T, const uint8_t *cls, const ChildSexes sex, uint8_t *calls) {
  constexpr uint32_t NC = NS - 2;
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_items) return;
  const uint32_t v = t / NC, ch = t % NC;
  const uint32_t cs = ch == 0 ? 0 : ch + 2;  // DKB_CHILD_SAMPLE
  const uint32_t *h = hits + (size_t)v * 2 * NS, *d = distinct + (size_t)v * 2 * NS;  // [allele*NS+sample]
  const uint32_t m = parent_clauses(cls ? cls[v] : (uint32_t)DKB_LOCUS_AUTOSOMAL, (sex >> (2 * ch)) & 3u);
  uint8_t c = 0;
  if (h[NS + cs] < T.min_child_alt_hits || d[NS + cs] < T.min_child_alt_distinct) c |= DKB_CALL_CHILD_LOW;
  if ((m & 1) && h[NS + 1] > T.max_parent_alt_hits) c |= DKB_CALL_MOTHER_ALT;
  if ((m & 2) && h[NS + 2] > T.max_parent_alt_hits) c |= DKB_CALL_FATHER_ALT;
  if (((m & 1) && h[1] < T.min_parent_ref_hits) || ((m & 2) && h[2] < T.min_parent_ref_hits))
    c |= DKB_CALL_PARENT_UNCOVERED;
  if (m & 4) c |= DKB_CALL_NO_COPY;
  calls[t] = c ? c : DKB_CALL_DENOVO;
}

}  // namespace dkb

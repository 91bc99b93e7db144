// dkb_scan.cuh — kernel 2: streaming extract-and-probe over a packed read
// stream (the GPU form of src/kmer.rs's per-read k-mer iteration feeding
// src/counter.rs's membership counting; both unmounted, DESIGN.md §2 is the spec).
//
// Every stream position p with p % D == 0 has its s-mer tested against a
// seed filter held in shared memory — or, for very large candidate tables, in
// L2 — (stage A, the only per-position work).
// Filter hits are verified against the exact seed table in L2 with ONE 4-byte load each,
// looked at one tile later (stage B).  At strides 2 and 4 every lane verifies its own hits
// in up to four rounds per tile; at the other strides the hits are compacted per (macro)
// tile and verified 32 at a time.  A verified seed has a 32-byte record: the offsets j at
// which some table key designates it, and what those keys look like around the seed.  The
// read is compared with that neighbourhood once; each window w = p - j inside the matching
// run is canonicalised and probed in the key table, one window per lane (stage C).  A slot
// is counted only when its own designated offset for class (j % D) equals j, so a matching
// window is counted exactly once however many seeds it contains (proof in DESIGN.md §4).
// A direct record (an isolated SNV's seed, dkb_device.cuh) names its windows' entries itself:
// its windows are counted in phase 1 without the key table.
#pragma once
#include "dkb_device.cuh"

namespace dkb {

// FM = filter mode (dkb_device.cuh): 0 seed filter in shared memory, 1 in L2, 2 in L2 behind a
// one-bit shared-memory pre-filter, 3 / 4 = 1 / 2 with gated lookups.
// RG = region mode (DESIGN.md §2): a window counts toward an entry only when its read's
// alignment interval overlaps the entry's variant window.
template <int D, int NH, int FM, bool PROF, bool RG>
struct ScanWarp {
  static constexpr bool GF = FM > 0, PRE = fm_pre(FM), GATE = fm_gate(FM);
  static constexpr int HL_CAP = hl_cap(FM);
  static constexpr bool CANON = canon_for_mode(FM);  // seeds keyed by min(s-mer, its reverse complement)
  // Strides 8 and 16 leave 8 / 4 lookups per lane in a 2048-position tile; SUB such tiles
  // form a macro tile with 32 lookups per lane so that hit handling and loop overhead are
  // paid once per macro tile.
  static constexpr bool MACRO = D >= 8;
  static constexpr int LPT = 64 / D;                 // lookups per lane and (sub-)tile
  static constexpr int SUB = MACRO ? 32 / LPT : 1;   // sub-tiles per macro tile
  static constexpr bool LOCAL = D == 2 || D == 4;    // lane-local hit verification
  const ScanParams &P;
  int cur = 0;  // segment (packed stream) the warp is working on; its fields are read from
                // the parameter block where needed rather than held in registers
  const uint32_t *filt;
  uint16_t *hl;  // filter-hit ids of the current tile: lane << 6 | lookup index
  uint64_t *cq;  // ring of verified seeds: seed-table slot << 32 | position
  uint32_t ch = 0, ct = 0;
  int lane;
  uint32_t lt_mask;
  uint64_t keep = l2_policy_evict_last();  // cache policy of every filter and table load
  const uint32_t zero;                     // 0, but not to the compiler
  const uint32_t fbase;                    // shared-memory address of the (pre-)filter
  // stage B probes in flight (issued at the end of one tile, consumed in the next)
  uint32_t pend_n = 0, pend_x = 0, pend_p = 0, pend_b = 0, pend_v = 0, pend_f = 0;
  unsigned long long n_bloom = 0, n_seed = 0, n_probe = 0, n_hit = 0;

  __device__ __forceinline__ ScanWarp(const ScanParams &p, const uint32_t *f, uint16_t *h,
                                      uint64_t *c, int l)
      : P(p), filt(f), hl(h), cq(c), lane(l), lt_mask((1u << l) - 1), zero(p.four >> 3),
        fbase((uint32_t)__cvta_generic_to_shared(f)) {}

  __device__ __forceinline__ uint32_t ld_bases(uint32_t wi) const {
    return wi < P.seg[cur].n_bwords ? __ldg(P.seg[cur].bases + wi) : 0u;
  }
  __device__ __forceinline__ uint32_t ld_mask(uint32_t wi) const {
    return wi < P.seg[cur].n_mwords ? __ldg(P.seg[cur].mask + wi) : 0u;
  }

  // ---- region mode: the read that holds stream position p --------------------------
  // The last read starting at or before p, searched between the hints of p's tile and the
  // next one (a tile holds about 14 reads of 150 bases: four steps).  p is a position of
  // segment `cur`, whose hints are read here: stage C only sees seeds of `cur`, because a warp
  // drains every pending probe and verified seed (drain()) before it moves to another segment.
  __device__ __forceinline__ uint32_t find_read(uint32_t p) const {
    // (no min() here: naming it in this class changes how the whole-stream kernels compile)
    const uint32_t nt = P.rseg[cur].n_tiles;
    uint32_t t = p >> LOCI_TILE_SHIFT;
    if (t >= nt) t = nt - 1;
    const uint32_t *const hint = P.tile_read + P.rseg[cur].tile_base + t;
    uint32_t a = __ldg(hint), b = __ldg(hint + 1);
    while (a < b) {
      const uint32_t mid = b - (b - a) / 2;
      if (__ldg(P.read_start + mid) <= p) a = mid; else b = mid - 1;
    }
    return a;
  }
  // Region mode: may read rd count toward entry e?  Only key-table matches get here.
  __device__ __forceinline__ bool in_region(uint32_t rd, uint32_t e) const {
    if constexpr (RG) return spans_overlap(__ldg(P.read_span + rd), __ldg(P.entry_win + e));
    else return true;
  }

  // ---- stage C: the candidate windows of up to n verified seeds --------------------
  // Key-table probe of one window: v = its k bases in stream order (first base least
  // significant), j = the offset at which it would designate the seed that led here,
  // rd = the read it lies in (region mode only).
  __device__ __forceinline__ void probe_window(uint64_t v, int j, uint32_t rd) {
    const int k = P.k;
    const uint64_t km = kmer_mask(k);
    if (PROF) n_probe++;
    const uint64_t fwd = base_reverse(v, k);
    const uint64_t rc = ~v & km;  // complement of the stream-order value IS the rc key
    const uint64_t key = fwd <= rc ? fwd : rc;
    const int ori = fwd <= rc ? 0 : 1;
    uint32_t bk = key_bucket(key, P.kt.bucket_mask);
    uint32_t *const counts = P.seg[cur].counts;
    while (true) {
      const uint4 *bp = P.kt.slots + bk * KBUCKET;
      const uint4 s0 = ldg_v4_hint(bp, keep), s1 = ldg_v4_hint(bp + 1, keep);
      const uint64_t k0 = slot_key(s0), k1 = slot_key(s1);
      if (k0 == key && s0.z != ENTRY_DEAD && slot_offset(s0.w, ori, j % D, D) == (uint32_t)j) {
        if (in_region(rd, s0.z)) atomicAdd(counts + s0.z, 1u);
        if (PROF) n_hit++;
      }
      if (k1 == key && s1.z != ENTRY_DEAD && slot_offset(s1.w, ori, j % D, D) == (uint32_t)j) {
        if (in_region(rd, s1.z)) atomicAdd(counts + s1.z, 1u);
        if (PROF) n_hit++;
      }
      if (k0 == KEY_EMPTY || k1 == KEY_EMPTY) break;  // bucket not full: nothing spilled
      bk = (bk + 1) & P.kt.bucket_mask;
    }
  }

  // Phase 1, one lane per verified seed.  All windows of a seed at p lie in
  // [p - (k - s), p + k): their bases and mask bits are fetched once (5 + 3 words) together
  // with the seed's number; then the seed's record (SeedRec, one 32-byte sector) says which
  // offsets are designated and what the designating keys look like around the seed.  The
  // read is compared with that neighbourhood once, invalid positions count as mismatches,
  // and only windows inside the matching run around the seed survive.  A chance seed match
  // (the common case on unrelated sequence) ends here.
  // Phase 2, one lane per surviving window: the owners list (lane, offset) pairs in the ring
  // slots just consumed, and the warp probes them 32 at a time - a seed's ~16 windows no
  // longer cost one dependent L2 round trip each inside a single lane.
  // Region mode resolves the seed's read once here: a counted window contains the seed and
  // no separator, so it lies in the seed's read; phase 2 takes it from the owner lane.
  // A direct record's windows are counted in phase 1 and leave no tasks for phase 2.
  __device__ __forceinline__ void stage_c(uint32_t n) {
    const int k = P.k, s = P.s, E = k - s;
    const uint64_t km = kmer_mask(k);
    uint32_t info = 0, p = 0, rn0 = 0, rn1 = 0, rn2 = 0;
    uint32_t rd = 0;  // region mode: the seed's read
    const uint32_t n_pos = P.seg[cur].n_pos;
    if ((uint32_t)lane < n) {
      const uint64_t e = cq[(ch + lane) & (CQ_CAP - 1)];
      p = (uint32_t)e;
      const uint32_t start = p > (uint32_t)E ? p - (uint32_t)E : 0u;
      const uint32_t bw0 = start >> 4, mw0 = start >> 5;
      // the record for this read orientation: a 32-byte half of the seed's slot (half 0 is
      // the sector stage B already touched)
      const uint4 *rp = P.st.slots + 2 * (size_t)(uint32_t)(e >> 32);  // e >> 32 = 2 * slot + flip
      const uint4 r0 = ldg_v4_hint(rp, keep), r1 = ldg_v4_hint(rp + 1, keep);
      const uint32_t nb0 = r0.z, nb1 = r0.w, nb2 = r1.x;
      uint32_t wd0 = r1.y, wd1 = r1.z, wd2 = r1.w;
      uint32_t b[5], m[3];
#pragma unroll
      for (int i = 0; i < 5; i++) b[i] = ld_bases(bw0 + i);
#pragma unroll
      for (int i = 0; i < 3; i++) m[i] = ld_mask(mw0 + i);
      info = r0.y & INFO_OFFSETS;
      const bool direct = (r0.y & INFO_DIRECT) != 0;
      if (p >= (uint32_t)E && E + k <= NB_BASES) {
        if (direct) {
          // a direct record's wild mask: the bases no designated window covers (window j covers
          // [E - j, E - j + k)), and X
          const int lo = 2 * (E - (31 - __clz(info))), hi = 2 * (E + k - (__ffs(info) - 1));
          const unsigned __int128 one = 1;
          const unsigned __int128 wild =
              ~(((one << hi) - 1) ^ ((one << lo) - 1)) | (unsigned __int128)3 << (2 * (r1.w & 63));
          wd0 = (uint32_t)wild;
          wd1 = (uint32_t)(wild >> 32);
          wd2 = (uint32_t)(wild >> 64);
        }
        // the read's neighbourhood (base 0 = p - E) and its mismatches, 2 bits per base
        const uint32_t sh = 2 * (start & 15);
        rn0 = __funnelshift_r(b[0], b[1], sh);
        rn1 = __funnelshift_r(b[1], b[2], sh);
        rn2 = __funnelshift_r(b[2], b[3], sh);
        const uint32_t mm0 = (rn0 ^ nb0) & ~wd0, mm1 = (rn1 ^ nb1) & ~wd1, mm2 = (rn2 ^ nb2) & ~wd2;
        const unsigned __int128 mm = (unsigned __int128)mm2 << 64 | (unsigned __int128)mm1 << 32 | mm0;
        // invalid positions (N, low quality, read separators, end of stream), 1 bit per base
        const uint32_t mo = start & 31;
        uint64_t inv = ~((uint64_t)__funnelshift_r(m[1], m[2], mo) << 32 | __funnelshift_r(m[0], m[1], mo));
        // end of stream: nothing at or beyond n_pos is a base, whatever the padding bits say
        if (start >= n_pos) inv = ~0ull;
        else if (n_pos - start < (uint32_t)NB_BASES) inv |= ~0ull << (n_pos - start);
        inv &= (1ull << NB_BASES) - 1;
        // R = first bad base at or after the seed's end, Lm = last one before its start; nothing
        // beyond base E + k is covered by a window, so both searches fit 64 bits
        const uint64_t ma = (uint64_t)(mm >> (2 * (E + s))), mb = (uint64_t)mm & ((1ull << (2 * E)) - 1);
        const uint64_t ia = inv >> (E + s), ib = inv & ((1ull << E) - 1);
        int R = NB_BASES, Lm = -1;
        if (ma) R = E + s + ((__ffsll((long long)ma) - 1) >> 1);
        if (ia) R = min(R, E + s + __ffsll((long long)ia) - 1);
        if (mb) Lm = (63 - __clzll((long long)mb)) >> 1;
        if (ib) Lm = max(Lm, 63 - __clzll((long long)ib));
        // window j covers bases [E - j, E - j + k): inside (Lm, R)  <=>  E + k - R <= j < E - Lm
        const int jlo = E + k - R > 0 ? E + k - R : 0, jhi = E - Lm - 1;
        info = jhi >= jlo ? info & ((2u << jhi) - 1u) & ~((1u << jlo) - 1u) : 0u;
        if ((inv >> E) & ((1ull << s) - 1)) info = 0;  // an invalid base inside the seed itself
        // Direct record: a window left here equals the key of allele a's designation at its offset
        // j exactly when the read's base at X is one allele a shows there (DESIGN.md §4), and that
        // key's only live entry is c_a + sigma_a * j: count it here, no key-table probe.
        const uint32_t x = r1.w & 63;
        const uint32_t rb = ((x < 16 ? rn0 : x < 32 ? rn1 : rn2) >> (2 * (x & 15))) & 3;
        const bool a1 = (r1.w >> (DIR_PICK1 + rb)) & 1;
        if (PROF && direct) n_probe += __popc(info);  // the windows the key table would have been asked about
        if (direct && !a1 && !((r1.w >> (DIR_PICK0 + rb)) & 1)) info = 0;
        if constexpr (RG) {
          if (info) rd = find_read(p);  // (a chance seed match needs no read)
        }
        if (direct) {
          const uint32_t c = a1 ? r1.z : r1.y;
          const bool neg = (r1.w >> (a1 ? DIR_NEG1 : DIR_NEG0)) & 1;
          uint32_t *const counts = P.seg[cur].counts;
          while (info) {
            const uint32_t j = __ffs(info) - 1;
            info &= info - 1;
            const uint32_t e = neg ? c - j : c + j;
            if (in_region(rd, e)) atomicAdd(counts + e, 1u);
            if (PROF) n_hit++;
          }
        }
      } else {
        // no usable neighbourhood (stream start, or 2k - s > NB_BASES): every designated
        // offset is checked here, one after the other
        const uint32_t vm = (1u << k) - 1;  // k <= 31
        if constexpr (RG) rd = find_read(p);
        while (info) {
          const int j = __ffs(info) - 1;
          info &= info - 1;
          if (p < (uint32_t)j) continue;
          const uint32_t w = p - (uint32_t)j;
          if (w + (uint32_t)k > n_pos) continue;
          const uint32_t wo = w - (mw0 << 5);  // < 64
          const uint32_t mbits = wo < 32 ? __funnelshift_r(m[0], m[1], wo)
                                         : __funnelshift_r(m[1], m[2], wo - 32);
          if ((mbits & vm) != vm) continue;
          const uint32_t bo = w - (bw0 << 4);  // < 48
          uint32_t x0 = b[0], x1 = b[1], x2 = b[2];
          if (bo >= 16) { x0 = b[1]; x1 = b[2]; x2 = b[3]; }
          if (bo >= 32) { x0 = b[2]; x1 = b[3]; x2 = b[4]; }
          const uint32_t sh = 2 * (bo & 15);
          probe_window(((uint64_t)__funnelshift_r(x1, x2, sh) << 32 | __funnelshift_r(x0, x1, sh)) & km, j, rd);
        }
      }
    }
    // ---- phase 2 ----
    if (!__any_sync(FULL_MASK, info != 0)) {  // every window was counted in phase 1, or none survived
      ch += n;
      __syncwarp();
      return;
    }
    uint32_t cnt = __popc(info), incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(FULL_MASK, incl, o);
      if (lane >= o) incl += t;
    }
    const uint32_t total = __shfl_sync(FULL_MASK, incl, 31);
    uint16_t *tl = reinterpret_cast<uint16_t *>(cq);  // task t lives in consumed ring slot ch + t / 4
    constexpr uint32_t TL_CAP = 128;                  // 32 slots of 8 bytes
    for (uint32_t base = 0; base < total; base += TL_CAP) {
      uint32_t idx = incl - cnt - base;  // wraps below zero for tasks of earlier passes
      uint32_t a = info;
      while (a) {
        const int j = __ffs(a) - 1;
        a &= a - 1;
        if (idx < TL_CAP) tl[((ch + (idx >> 2)) & (CQ_CAP - 1)) * 4 + (idx & 3)] = (uint16_t)(lane << 5 | j);
        idx++;
      }
      __syncwarp();
      const uint32_t here = min(total - base, TL_CAP);
      for (uint32_t r = 0; r < here; r += 32) {
        const uint32_t t = r + lane;
        const bool act = t < here;
        const uint32_t task = act ? tl[((ch + (t >> 2)) & (CQ_CAP - 1)) * 4 + (t & 3)] : 0u;
        const int src = task >> 5, j = task & 31;
        const uint32_t q0 = __shfl_sync(FULL_MASK, rn0, src), q1 = __shfl_sync(FULL_MASK, rn1, src),
                       q2 = __shfl_sync(FULL_MASK, rn2, src);
        uint32_t qr = 0;
        if constexpr (RG) qr = __shfl_sync(FULL_MASK, rd, src);
        if (act) {
          const int o = E - j;  // first base of the window in the neighbourhood, 0 .. E
          const uint32_t x0 = o < 16 ? q0 : q1, x1 = o < 16 ? q1 : q2, x2 = o < 16 ? q2 : 0u;
          const uint32_t sh = 2 * (o & 15);
          probe_window(((uint64_t)__funnelshift_r(x1, x2, sh) << 32 | __funnelshift_r(x0, x1, sh)) & km, j, qr);
        }
      }
      __syncwarp();
    }
    ch += n;
    __syncwarp();
  }

  // ---- stage B helpers ------------------------------------------------------------
  // ptxas puts every global load of the loop on one scoreboard, so the first use of the
  // prefetched next tile would also wait for whatever table loads were issued after it -
  // a full L2 round trip per tile.  Settle the prefetch (issued a whole stage A ago) BEFORE
  // issuing table loads: the empty asm makes its words plain register values from here on.
  __device__ __forceinline__ static void settle(uint32_t (&r)[5]) {
    asm volatile("" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]));
  }

  // s-mer (masked) -> the seed it is stored under, and whether that is its reverse complement
  __device__ __forceinline__ uint32_t canon(uint32_t x, uint32_t &flip) const {
    if constexpr (CANON) return seed_canon(x, P.cshift, flip);
    flip = 0;
    return x;
  }

  // Stage B checks a seed against the probe array in the shared-memory filter mode and
  // against the slot table itself in the L2 modes (dkb_device.cuh, SeedTable).
  static constexpr bool PROBE = FM == 0;
  __device__ __forceinline__ bool use_probe() const { return PROBE && P.st.n_probe != 0; }
  __device__ __forceinline__ uint32_t vhome(uint32_t x) const {
    return seed_home(x, use_probe() ? P.st.n_probe : P.st.n_slots);
  }
  // the word that says whether entry `e` holds a seed (and whether to walk on)
  __device__ __forceinline__ uint32_t ld_slot_word(uint32_t e) const {
    if (use_probe()) return ldg_u32_hint(P.st.probe + e, keep);
    return ldg_u32_hint(reinterpret_cast<const uint32_t *>(P.st.slots) + 16 * (size_t)e, keep);
  }
  // entry of the structure stage B verified against -> the seed's slot
  __device__ __forceinline__ uint32_t slot_of(uint32_t x, uint32_t e) const {
    if (!use_probe()) return e;
    uint32_t b = seed_home(x, P.st.n_slots);
    while ((ldg_u32_hint(reinterpret_cast<const uint32_t *>(P.st.slots) + 16 * (size_t)b, keep) & ST_SEED_BITS) != x)
      b = seed_next(b, P.st.n_slots);
    return b;
  }

  // Slow half of a seed-table lookup: the home slot holds another seed and carries
  // ST_MOVED_BIT, so the seed may sit further along (linear probing, ends at a free slot).
  __device__ __forceinline__ bool walk(uint32_t x, uint32_t &slot) const {
    uint32_t b = slot;
    const uint32_t n = use_probe() ? P.st.n_probe : P.st.n_slots;
    while (true) {
      b = seed_next(b, n);
      const uint32_t v = ld_slot_word(b);
      if ((v & ST_SEED_BITS) == x) {
        slot = b;
        return true;
      }
      if (v & ST_FREE_BIT) return false;
    }
  }

  // Queue the lanes' verified seeds (2 * seed-table slot + read orientation, stream position) for stage C.
  __device__ __forceinline__ void push_verified(bool found, uint32_t slot, uint32_t p) {
    const uint32_t bal = __ballot_sync(FULL_MASK, found);
    if (bal == 0) return;
    if (found) cq[(ct + __popc(bal & lt_mask)) & (CQ_CAP - 1)] = (uint64_t)slot << 32 | p;
    ct += __popc(bal);
    if (PROF && found) n_seed++;
    __syncwarp();
    if (ct - ch >= 32) stage_c(32);
  }

  // ---- stage B, lane-local form (strides 2 and 4) -----------------------------------
  // Every lane verifies its OWN filter hits: no compaction, no shuffles, no id list.  Round
  // r takes the lane's r-th hit of the tile, cuts its seed out of the lane's registers and
  // issues the 4-byte load of the seed's home slot; the loads are looked at one tile later
  // (after the next stage A), so L2 latency hides inside the warp.  A tile has ~1 hit per
  // lane, the busiest lane 3-4; lanes beyond NR hits (rare) finish synchronously.
  static constexpr int NR = 4;
  uint32_t lv[NR] = {ST_EMPTY, ST_EMPTY, ST_EMPTY, ST_EMPTY};  // loaded home-slot words
  uint32_t lx[NR] = {0, 0, 0, 0};                              // their seeds
  uint32_t lidx = 0, lbase = 0;  // hit-mask bit of round r in byte r; the tile's first position

  // Seed of the lookup whose hit bit is bit b of the tile's mask (lookup i = 31 - b starts
  // i * D positions into the lane's chunk).
  __device__ __forceinline__ uint32_t cut_seed(const uint32_t (&w)[5], uint32_t b) const {
    constexpr uint32_t HI = D == 4 ? 8u : 16u, LO = D == 4 ? 4u : 8u;  // bits of b above the word index
    // word index c = ((31 - b) * D) >> 4, taken from the inverted bits of b
    uint32_t a0 = w[2], a1 = w[3], a2 = w[4];
    if (b & HI) { a0 = w[0]; a1 = w[1]; a2 = w[2]; }
    uint32_t lo = a1, hi = a2;
    if (b & LO) { lo = a0; hi = a1; }
    // shift = 2 * ((31 - b) * D mod 16) = (62 D - 2 D b) mod 32: the funnel shift wraps
    return __funnelshift_r(lo, hi, 62u * D - 2u * D * b) & P.seed_mask;
  }

  // after = a value computed by the work that must come BEFORE the loaded words are looked
  // at (the hit mask of the stage A that ran meanwhile).  The comparison mask is made to
  // depend on it through a run-time zero; otherwise ptxas hoists these compares to the top
  // of that stage A, where they wait for the scoreboard of loads issued a moment earlier.
  __device__ __forceinline__ void resolve_local(uint32_t after) {
    const uint32_t msk = ST_SEED_BITS + (after & zero);  // a sum: no known bits to split off
    // bit r: round r's slot holds the seed, or says the seed may have moved on
    uint32_t mm = 0;
#pragma unroll
    for (int r = 0; r < NR; r++)
      mm |= (uint32_t)(((lv[r] ^ lx[r]) & msk) == 0 || (lv[r] & ~msk) != 0) << r;
    if (!__any_sync(FULL_MASK, mm != 0)) return;
    // About every second tile (a true seed somewhere in the warp).  One rolled copy of the
    // code: each lane takes its lowest flagged round, whichever that is.
    do {
      const bool has = mm != 0;
      const int r = has ? __ffs(mm) - 1 : 0;
      mm &= mm - 1;
      uint32_t v = lv[0], x = lx[0];
      if (r == 1) { v = lv[1]; x = lx[1]; }
      if (r == 2) { v = lv[2]; x = lx[2]; }
      if (r == 3) { v = lv[3]; x = lx[3]; }
      const uint32_t i = 31u - ((lidx >> (8 * r)) & 31u), flip = (lidx >> (8 * r + 7)) & 1u;
      bool found = has && ((v ^ x) & ST_SEED_BITS) == 0;
      const bool moved = has && !found;  // flagged without a match: ST_MOVED_BIT
      uint32_t slot = vhome(x);
      if (__any_sync(FULL_MASK, moved)) {
        if (moved) found = walk(x, slot);
        __syncwarp();
      }
      if (found) slot = slot_of(x, slot);
      push_verified(found, 2 * slot + flip, lbase + lane * CHUNK + i * D);
    } while (__any_sync(FULL_MASK, mm != 0));
  }

  // Start the rounds of the tile whose words are w and whose hit mask is acc (bit 31 =
  // lookup 0).  Any earlier rounds must have been resolved.
  __device__ __forceinline__ void start_local(uint32_t acc, const uint32_t (&w)[5],
                                              uint32_t tile_base) {
#pragma unroll
    for (int r = 0; r < NR; r++) lv[r] = ST_EMPTY;
    if (PROF) n_bloom += __popc(acc);
    uint32_t a = acc;  // bit 31 = lookup 0
    lbase = tile_base;
    while (true) {
      lidx = 0;
#pragma unroll
      for (int r = 0; r < NR; r++) {
        if (!__any_sync(FULL_MASK, a != 0)) break;
        const bool has = a != 0;
        const uint32_t b = 31u - __clz(a);  // any hit will do: take the highest bit
        a &= ~(1u << (b & 31));
        uint32_t flip;
        const uint32_t x = canon(cut_seed(w, b), flip);
        lx[r] = x;
        if (has) lv[r] = ld_slot_word(vhome(x));
        lidx |= ((b & 31) | flip << 7) << (8 * r);
      }
      if (!__any_sync(FULL_MASK, a != 0)) break;
      // a lane with more than NR hits in one tile (rare): finish these rounds now
      resolve_local(a);
#pragma unroll
      for (int r = 0; r < NR; r++) lv[r] = ST_EMPTY;
    }
  }

  // ---- stage B, batch form (strides 1, 8, 16), second half: use the slots loaded one
  // batch ago
  // (after: see resolve_local)
  __device__ __forceinline__ void consume_pending(uint32_t after) {
    if (pend_n == 0) return;
    const bool act = (uint32_t)lane < pend_n;
    const uint32_t msk = ST_SEED_BITS + (after & zero);
    const uint32_t v = pend_v, x = pend_x;
    bool found = act && ((v ^ x) & msk) == 0;
    const bool moved = act && !found && (v & ~msk) != 0;
    uint32_t slot = pend_b;
    if (__any_sync(FULL_MASK, moved)) {
      if (moved) found = walk(x, slot);
      __syncwarp();
    }
    pend_n = 0;
    if (found) slot = slot_of(x, slot);
    push_verified(found, 2 * slot + pend_f, pend_p);
  }

  // ---- stage B, batch form, first half: start the exact check of hits [first, first + n)
  // Each lane takes one hit id, pulls the 16 bases at that position out of the
  // owning lane's registers with shuffles (no trip back to L2) and issues the
  // load of the seed's home slot.  tile_base = stream position of lane 0's chunk.
  __device__ __forceinline__ void issue_probes(uint32_t first, uint32_t n, const uint32_t (&w)[5],
                                               uint32_t tile_base) {
    const bool act = (uint32_t)lane < n;
    const uint32_t id = act ? hl[first + lane] : (uint32_t)lane << 6;
    const int src = id >> 6;
    pend_v = ST_EMPTY;
    if constexpr (MACRO) {
      // macro tiles (strides 8, 16): the lookup index runs over SUB sub-tiles whose words
      // are no longer in registers; hits are rare here, so re-read them from L2
      const uint32_t idx = id & 63;
      pend_p = tile_base + (idx / LPT) * WTILE + src * CHUNK + (idx % LPT) * D;
      const uint32_t wi = pend_p >> 4;
      pend_x = canon(__funnelshift_r(ld_bases(wi), ld_bases(wi + 1), 2 * (pend_p & 15)) & P.seed_mask, pend_f);
      pend_b = vhome(pend_x);
      if (act) pend_v = ld_slot_word(pend_b);
      pend_n = n;
      return;
    }
    const uint32_t q = (id & 63) * D;  // offset inside the owning lane's chunk
    const uint32_t c = q >> 4;
    uint32_t v[5];
#pragma unroll
    for (int i = 0; i < 5; i++) v[i] = __shfl_sync(FULL_MASK, w[i], src);
    uint32_t lo = v[0], hi = v[1];
    if (c == 1) { lo = v[1]; hi = v[2]; }
    if (c == 2) { lo = v[2]; hi = v[3]; }
    if (c == 3) { lo = v[3]; hi = v[4]; }
    pend_x = canon(__funnelshift_r(lo, hi, 2 * (q & 15)) & P.seed_mask, pend_f);
    pend_p = tile_base + src * CHUNK + q;
    pend_b = vhome(pend_x);
    if (act) pend_v = ld_slot_word(pend_b);
    pend_n = n;
  }

  // ---- compact this tile's filter hits and start their verification ---------------
  // bit 31 of acc0 is lookup 0; acc1 (D == 1 only) continues at lookup 32.
  __device__ __forceinline__ void handle_hits(uint32_t acc0, uint32_t acc1,
                                              const uint32_t (&w)[5], uint32_t tile_base) {
    const uint32_t cnt = __popc(acc0) + (D == 1 ? __popc(acc1) : 0);
    if (PROF) n_bloom += cnt;
    // Exclusive prefix sum of the per-lane hit counts.  Counts are almost always
    // below 8, so three ballots of their bit planes replace five dependent shuffles.
    const uint32_t b0 = __ballot_sync(FULL_MASK, cnt & 1), b1 = __ballot_sync(FULL_MASK, cnt & 2),
                   b2 = __ballot_sync(FULL_MASK, cnt & 4), bhi = __ballot_sync(FULL_MASK, cnt > 7);
    if ((b0 | b1 | b2 | bhi) == 0) return;
    uint32_t total, excl;
    if (bhi == 0) {
      total = __popc(b0) + 2 * __popc(b1) + 4 * __popc(b2);
      excl = __popc(b0 & lt_mask) + 2 * __popc(b1 & lt_mask) + 4 * __popc(b2 & lt_mask);
    } else {
      uint32_t incl = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL_MASK, incl, o);
        if (lane >= o) incl += t;
      }
      total = __shfl_sync(FULL_MASK, incl, 31);
      excl = incl - cnt;
    }
    const uint32_t tag = (uint32_t)lane << 6;
    if constexpr (!MACRO) {
      if (total <= (uint32_t)HL_CAP) {
        // common case: the whole tile fits the id list, no bounds checks
        uint32_t idx = excl;
        uint32_t a = acc0;
        while (a) {
          const int i = __clz(a);
          a ^= 0x80000000u >> i;
          hl[idx++] = (uint16_t)(tag + i);
        }
        if (D == 1) {
          a = acc1;
          while (a) {
            const int i = __clz(a);
            a ^= 0x80000000u >> i;
            hl[idx++] = (uint16_t)(tag + 32 + i);
          }
        }
        __syncwarp();
        for (uint32_t r = 0; r < total; r += 32) {
          consume_pending(0);  // at most one batch of probes in flight
          issue_probes(r, min(total - r, 32u), w, tile_base);
        }
        __syncwarp();
        return;
      }
    }
    // the id list holds HL_CAP hits; denser tiles (low-complexity sequence) take more passes
    for (uint32_t base = 0; base < total; base += HL_CAP) {
      uint32_t idx = excl - base;  // wraps below zero for hits of earlier passes
      uint32_t a = acc0;
      while (a) {
        const int i = __clz(a);
        a ^= 0x80000000u >> i;
        if (idx < (uint32_t)HL_CAP) hl[idx] = (uint16_t)(tag + i);
        idx++;
      }
      if (D == 1) {
        a = acc1;
        while (a) {
          const int i = __clz(a);
          a ^= 0x80000000u >> i;
          if (idx < (uint32_t)HL_CAP) hl[idx] = (uint16_t)(tag + 32 + i);
          idx++;
        }
      }
      __syncwarp();
      const uint32_t here = min(total - base, (uint32_t)HL_CAP);
      for (uint32_t r = 0; r < here; r += 32) {
        consume_pending(0);  // at most one batch of probes in flight
        issue_probes(r, min(here - r, 32u), w, tile_base);
      }
      __syncwarp();
    }
  }

  __device__ __forceinline__ void drain() {
    if constexpr (LOCAL) resolve_local(0); else consume_pending(0);
    while (ct != ch) stage_c(min(ct - ch, 32u));
  }

  // bit * 2^e + a as ONE multiply-add (in C the compiler, knowing bit is 0 or 1, makes it a
  // compare, a select and an add - three ALU-pipe instructions)
  __device__ __forceinline__ uint32_t mad_pw(uint32_t bit, int e, uint32_t a) const {
    uint32_t r;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(bit), "r"(P.pw[e]), "r"(a));
    return r;
  }

  // One filter lookup of the s-mer whose bases start at the low bits of x: 1 when every
  // filter bit of x is set (layout: bloom_bits() in dkb_device.cuh).  Issue cost on sm_100
  // (scripts/micro/int_pipes.cu): ALU-pipe and FMA-pipe instructions take 2 cycles per warp
  // each and overlap; IMAD.WIDE 2.4; a multiply-high 5 and it holds up the ALU pipe, so
  // there is none here.  ALU: cut (caller), index shift, one shift per filter bit, AND.
  // FMA: hash, wide multiply, address, and the caller's accumulate.
  __device__ __forceinline__ uint32_t lookup(uint32_t x, uint32_t mult, bool ok = true) const {
    if constexpr (CANON) {
      uint32_t flip;
      x = seed_canon(x & P.seed_mask, P.cshift, flip);
    }
    const uint32_t h = x * mult;
    unsigned long long prod;  // forced wide: ptxas would turn a plain (u64)h * n >> 32 into IMAD.HI
    uint32_t word;
    asm("mul.wide.u32 %0, %1, %2;" : "=l"(prod) : "r"(h), "r"(P.filter_words));
    // byte address = idx * 4 + base as a multiply-add (P.four is opaque), not an ALU-pipe LEA
    const uint32_t addr = (uint32_t)(prod >> 32) * P.four + fbase;
    word = 0;
    if (ok) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(word) : "r"(addr));
    const uint32_t lo = (uint32_t)prod;
    uint32_t bit = __funnelshift_r(word, 0, x);  // the shift wraps: bit (x & 31) comes down to bit 0
    if (NH >= 2) bit &= __funnelshift_r(word, 0, lo >> 27);
    if (NH >= 3) bit &= __funnelshift_r(word, 0, lo >> 22);
    if (NH >= 4) bit &= __funnelshift_r(word, 0, lo >> 17);
    return bit & 1u;
  }

  // ---- L2 filter mode: N lookups at once, in three passes so that the N shared-memory loads
  // of the pre-filter, and then the N L2 loads behind it, are all in flight together (one
  // lookup at a time, each load's latency was exposed in full: the LDS 30 cycles, the L2 load
  // 300+, per lookup and warp).  x[i] = the s-mer of lookup first + i; returns a with the hit
  // bits added at bit positions top - (first + i).
  // ok bit i = the seed of lookup i holds only usable bases (stage A reads the flag stream for
  // this): a seed with an N, a low-quality base or a read separator inside cannot belong to a
  // countable window, so its lookup - the LDS and the L2 gather - is skipped.
  template <int N>
  __device__ __forceinline__ uint32_t gf_lookups(const uint32_t (&xr)[N], uint32_t ok, uint32_t a, int top) const {
    const uint32_t mult = P.seed_mult;
    uint32_t x[N];
#pragma unroll
    for (int i = 0; i < N; i++) {
      x[i] = xr[i];
      if constexpr (CANON) {
        uint32_t flip;
        x[i] = seed_canon(xr[i] & P.seed_mask, P.cshift, flip);
      }
    }
    uint32_t h[N], w1[N], s1[N];
    if constexpr (PRE) {
#pragma unroll
      for (int i = 0; i < N; i++) {
        h[i] = x[i] * mult;
        unsigned long long p1;
        asm("mul.wide.u32 %0, %1, %2;" : "=l"(p1) : "r"(h[i]), "r"(P.pre_words));
        // the bit inside the word comes from the hash too (top of the product's low half): the
        // raw low bits of a CANONICAL seed are skewed, and reads skew the same way - taking them
        // as the bit index let 49 % of the lookups through instead of the 41 % the fill predicts
        s1[i] = (uint32_t)p1 >> 27;
        w1[i] = 0;
        if ((ok >> i) & 1u)
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w1[i]) : "r"((uint32_t)(p1 >> 32) * P.four + fbase));
      }
    }
    uint32_t word[N], lo[N];
#pragma unroll
    for (int i = 0; i < N; i++) {
      const uint32_t hh = PRE ? h[i] * PRE_REHASH : x[i] * mult;
      unsigned long long prod;
      asm("mul.wide.u32 %0, %1, %2;" : "=l"(prod) : "r"(hh), "r"(P.bloom_words));
      lo[i] = (uint32_t)prod;
      word[i] = 0;
      bool pass = (ok >> i) & 1u;
      if constexpr (PRE) pass = (__funnelshift_r(w1[i], 0, s1[i]) & 1u) != 0;  // (w1 is 0 for a skipped lookup)
      // address = base + 4 * word index as ONE wide multiply-add
      unsigned long long ga;
      asm("mad.wide.u32 %0, %1, 4, %2;" : "=l"(ga) : "r"((uint32_t)(prod >> 32)), "l"(P.bloom));
      // (no L1 allocation: the filter is far larger than L1, and leaving L1 to the loads
      // that need it is worth 4 %; the same hint on stream or table loads costs 1-2 %)
      if (pass) {
        asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;"
                     : "=r"(word[i]) : "l"(ga), "l"(keep));
      }
    }
#pragma unroll
    for (int i = 0; i < N; i++) {
      uint32_t bit = __funnelshift_r(word[i], 0, x[i]);  // the shift wraps: bit (x & 31) comes down to bit 0
      if (NH >= 2) bit &= __funnelshift_r(word[i], 0, lo[i] >> 27);
      a = mad_pw(bit & 1u, top - i, a);
    }
    return a;
  }

  // ---- stage A, macro-tile form: LPT lookups of one sub-tile, hit bits in the low bits,
  // first lookup highest.  At stride 16 every seed lies inside one word (s <= 15): no
  // cut, no halo.
  // mk = the flags of the lane's 64 positions.  A seed that runs past them (stride 8, last
  // lookup of the chunk) is looked up regardless - skipping is only ever an optimisation.
  __device__ __forceinline__ uint32_t stage_a_sub(const uint32_t (&w)[5], uint2 mk) const {
    const uint32_t mult = P.seed_mult;
    const uint32_t sbits = (1u << P.s) - 1u;  // s <= 15
    uint32_t a = 0;
    uint32_t okm = ~0u;  // bit n = the seed of lookup n (at chunk position n * D) is usable throughout
    if constexpr (GATE && D == 16) {
      // two seeds per flag word (bits 0..s-1 and 16..16+s-1): all ones + 1 carries into bit s
      const uint32_t sel = sbits | sbits << 16;
      const uint32_t u0 = ((mk.x & sel) + 0x00010001u) >> P.s, u1 = ((mk.y & sel) + 0x00010001u) >> P.s;
      okm = (u0 & 1u) | (u0 >> 15 & 2u) | (u1 & 1u) << 2 | (u1 >> 13 & 8u);
    } else if constexpr (GATE) {
      okm = 0;
#pragma unroll
      for (int n = 0; n < LPT; n++) {
        const int pos = n * D;  // 0 .. 63
        uint32_t f;
        if (pos + 15 <= 32) f = mk.x >> pos;
        else if (pos >= 32 && pos + 15 <= 64) f = mk.y >> (pos - 32);
        else if (pos < 32) f = __funnelshift_r(mk.x, mk.y, pos);
        else f = mk.y >> (pos - 32) | ~0u << (64 - pos);  // the part beyond the chunk counts as usable
        okm |= (uint32_t)((f & sbits) == sbits) << n;
      }
    }
    if constexpr (GF) {
      constexpr int PERW = 16 / D;  // lookups per word (1 or 2)
#pragma unroll
      for (int c0 = 0; c0 < 4; c0 += 4 / PERW) {  // four lookups at a time
        uint32_t x[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int c = c0 + i / PERW, t = (i % PERW) * D;
          x[i] = t ? __funnelshift_r(w[c], w[c + 1], 2 * t) : w[c];
        }
        a = gf_lookups<4>(x, okm >> (c0 * PERW), a, LPT - 1 - c0 * PERW);
      }
      return a;
    }
    int n = 0;
#pragma unroll
    for (int c = 0; c < 4; c++) {
#pragma unroll
      for (int t = 0; t < 16; t += D, n++) {
        const uint32_t x = t ? __funnelshift_r(w[c], w[c + 1], 2 * t) : w[c];
        a = mad_pw(lookup(x, mult, (okm >> n) & 1u), LPT - 1 - n, a);
      }
    }
    return a;
  }

  // ---- stage A: the shared-memory seed filter over one lane chunk ---------------
  // w[0..3] hold this lane's 64 positions, w[4] the next 16 (halo for s-mers
  // that start in the chunk and end beyond it).
  __device__ __forceinline__ void stage_a(const uint32_t (&w)[5], uint32_t &acc0,
                                          uint32_t &acc1) const {
    const uint32_t mult = P.seed_mult;
    // Lookup n of the tile puts its hit bit at bit 31 - n of the mask (D == 1: of acc0 for
    // n < 32, of acc1 after) with a multiply-add by 2^(31 - n) from the parameter block -
    // the FMA pipe has the room, and a literal power of two would become an ALU-pipe shift.
    // Four chains, one per word.
    constexpr int NB = 16 / D;  // lookups per word
    uint32_t part[4];
#pragma unroll
    for (int c = 0; c < 4; c++) {
      uint32_t a = 0;
      if constexpr (GF) {  // strides 2 and 4: the word's 8 / 4 lookups, four at a time
#pragma unroll
        for (int t0 = 0; t0 < 16; t0 += 4 * D) {
          uint32_t x[4];
#pragma unroll
          for (int i = 0; i < 4; i++) {
            const int t = t0 + i * D;
            x[i] = t ? __funnelshift_r(w[c], w[c + 1], 2 * t) : w[c];
          }
          a = gf_lookups<4>(x, 0xFu, a, 31 - ((c * NB + t0 / D) & 31));
        }
      } else {
#pragma unroll
        for (int t = 0; t < 16; t += D) {
          const uint32_t x = t ? __funnelshift_r(w[c], w[c + 1], 2 * t) : w[c];
          const int n = (c * NB + t / D) & 31;
          a = mad_pw(lookup(x, mult), 31 - n, a);
        }
      }
      part[c] = a;
    }
    if constexpr (D == 1) {
      acc0 = part[0] + part[1];
      acc1 = part[2] + part[3];
    } else {
      acc0 = part[0] + part[1] + part[2] + part[3];
      acc1 = 0;
    }
  }
};

// ---- stream loads of the macro path ----------------------------------------------------
// Shared-memory filter mode: normal L2 priority - its filter hits are frequent and re-read
// their bases from L2 right after (evict-first costs 6 % at 250 candidates).  L2 filter modes:
// evict-first - hits are rare there, and the stream must not push the filter and the tables out.
template <int FM>
__device__ __forceinline__ uint4 ld_stream_v4(const uint32_t *p) {
  if (FM == 0) return __ldg(reinterpret_cast<const uint4 *>(p));
  return __ldcs(reinterpret_cast<const uint4 *>(p));
}

// tile -> registers.  Streaming (evict-first) loads: the stream is read once
// and must not push the seed / key tables out of L2.
__device__ __forceinline__ void load_tile(const ScanSegment &S, uint32_t tile, int lane,
                                          uint32_t (&w)[5]) {
  const uint32_t wi = tile * WTILE_WORDS + lane * 4;
  if (wi + 4 <= S.n_bwords) {
    const uint4 v = __ldcs(reinterpret_cast<const uint4 *>(S.bases + wi));
    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
  } else {
#pragma unroll
    for (int i = 0; i < 4; i++) w[i] = wi + i < S.n_bwords ? S.bases[wi + i] : 0u;
  }
  // w[4] of lane 31 = first word of the next warp tile; the other lanes get
  // theirs from lane + 1 in halo_finish(), AFTER the loads have landed, so the
  // prefetch of the next tile never stalls on a shuffle.
  w[4] = 0;
  if (lane == 31) w[4] = wi + 4 < S.n_bwords ? __ldg(S.bases + wi + 4) : 0u;
}

__device__ __forceinline__ void halo_finish(int lane, uint32_t (&w)[5]) {
  const uint32_t up = __shfl_down_sync(FULL_MASK, w[0], 1);
  if (lane != 31) w[4] = up;
}

// Work units (tiles, or macro tiles at strides 8 / 16) are numbered across the launch's
// segments; a warp takes units g, g + n_warps, ...  seg = the segment unit belongs to
// (n_seg once the units are used up).
struct UnitCursor {
  uint32_t unit;
  int seg;
  __device__ __forceinline__ void settle_seg(const ScanParams &P) {
    while (seg < P.n_seg && unit >= P.seg[seg].unit_end) seg++;
  }
  __device__ __forceinline__ bool live(const ScanParams &P) const { return seg < P.n_seg; }
  // index of the unit inside its segment
  __device__ __forceinline__ uint32_t local(const ScanParams &P) const {
    return unit - P.seg[seg].unit_begin;
  }
};

template <int D, int NH, int FM, bool PROF, bool RG>
__global__ void __launch_bounds__(SCAN_THREADS, 1) k_scan(const ScanParams P) {
  constexpr bool GF = FM > 0;
  extern __shared__ __align__(16) uint32_t smem[];
  uint32_t *filt = smem;
  uint64_t *cq_all = reinterpret_cast<uint64_t *>(smem + (GF ? P.pre_words : BLOOM_WORDS));
  uint16_t *hl_all = reinterpret_cast<uint16_t *>(cq_all + SCAN_WARPS * CQ_CAP);

  {
    const uint32_t n4 = (GF ? P.pre_words : (uint32_t)BLOOM_WORDS) / 4;
    const uint4 *src = reinterpret_cast<const uint4 *>(GF ? P.pre : P.bloom);
    for (uint32_t i = threadIdx.x; i < n4; i += SCAN_THREADS) reinterpret_cast<uint4 *>(filt)[i] = __ldg(src + i);
    __syncthreads();
  }

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int HL_CAP = hl_cap(FM);
  ScanWarp<D, NH, FM, PROF, RG> W(P, filt, hl_all + warp * HL_CAP, cq_all + warp * CQ_CAP, lane);

  const uint32_t n_warps = gridDim.x * SCAN_WARPS;
  UnitCursor c{warp * gridDim.x + blockIdx.x, 0};  // consecutive units on different SMs
  c.settle_seg(P);
  W.cur = c.live(P) ? c.seg : 0;
  if constexpr (ScanWarp<D, NH, FM, PROF, RG>::MACRO) {
    // Strides 8 / 16: a macro tile = SUB sub-tiles of 2048 positions (32 lookups per lane),
    // read in groups of GS sub-tiles (GS LDG.128 per lane in flight, 1-2 KB per warp), with
    // the next group prefetched while the current one is filtered.
    constexpr int SUB = ScanWarp<D, NH, FM, PROF, RG>::SUB, LPT = ScanWarp<D, NH, FM, PROF, RG>::LPT;
    constexpr int GS = MACRO_GS, GPM = SUB / GS;  // sub-tiles per group, groups per macro tile
    constexpr bool HALO = D < 16;          // at stride 16 every seed lies inside one word
    // a group that ends beyond the stream (the last one of a segment) is read word by word
    auto load_group_tail = [&](const ScanSegment &S, uint32_t t0, uint4 (&v)[GS], uint32_t &edge) {
      const uint32_t wb = t0 * WTILE_WORDS + lane * 4;
#pragma unroll
      for (int j = 0; j < GS; j++) {
        const uint32_t q = wb + j * WTILE_WORDS;
        v[j].x = q < S.n_bwords ? S.bases[q] : 0u;
        v[j].y = q + 1 < S.n_bwords ? S.bases[q + 1] : 0u;
        v[j].z = q + 2 < S.n_bwords ? S.bases[q + 2] : 0u;
        v[j].w = q + 3 < S.n_bwords ? S.bases[q + 3] : 0u;
      }
      const uint32_t e = (t0 + GS) * WTILE_WORDS;
      edge = HALO && e < S.n_bwords ? S.bases[e] : 0u;
    };
    // the flags of the lane's chunks in the group's sub-tiles: two words (64 positions) each
    constexpr bool GATE = fm_gate(FM);
    auto load_flags = [&](const ScanSegment &S, uint32_t t0, uint2 (&mk)[GS]) {
#pragma unroll
      for (int j = 0; j < GS; j++) {
        if constexpr (!GATE) {
          mk[j] = make_uint2(~0u, ~0u);
          continue;
        }
        const uint32_t mi = (t0 + j) * (WTILE / 32) + lane * 2;
        if (mi + 2 <= S.n_mwords) {
          mk[j] = __ldcs(reinterpret_cast<const uint2 *>(S.mask + mi));
        } else {
          mk[j].x = mi < S.n_mwords ? S.mask[mi] : 0u;
          mk[j].y = 0u;
        }
      }
    };
    // stage A of one group +, after the last group of a macro tile, its hit handling
    uint32_t acc = 0;
    auto filter_group = [&](const uint4 (&v)[GS], uint32_t edge, const uint2 (&mk)[GS]) {
#pragma unroll
      for (int j = 0; j < GS; j++) {
        uint32_t w[5] = {v[j].x, v[j].y, v[j].z, v[j].w, 0};
        if constexpr (HALO) {
          // lanes 0..30 take lane + 1's first word; lane 31 takes the first word of the
          // next sub-tile (lane 0's, or the group's edge word)
          const uint32_t up = __shfl_down_sync(FULL_MASK, w[0], 1);
          const uint32_t wrap = j + 1 < GS ? __shfl_sync(FULL_MASK, v[j + 1 < GS ? j + 1 : j].x, 0)
                                           : edge;
          w[4] = lane == 31 ? wrap : up;
        }
        acc = acc << LPT | W.stage_a_sub(w, mk[j]);
      }
    };
    auto load_group = [&](const ScanSegment &S, uint32_t t0, uint4 (&v)[GS], uint32_t &edge) {
      const uint32_t wb = t0 * WTILE_WORDS + lane * 4;
      if ((t0 + GS) * WTILE_WORDS + 4 <= S.n_bwords) {
#pragma unroll
        for (int j = 0; j < GS; j++) v[j] = ld_stream_v4<FM>(S.bases + wb + j * WTILE_WORDS);
        edge = 0;
        if (HALO && lane == 31) edge = __ldg(S.bases + (t0 + GS) * WTILE_WORDS);
      } else {  // the stream ends inside this group
        load_group_tail(S, t0, v, edge);
      }
    };
    int g = 0;
    uint4 nxt[GS];
    uint2 nxt_mk[GS];
    uint32_t nxt_edge = 0;
    if (c.live(P)) {
      load_group(P.seg[c.seg], c.local(P) * SUB, nxt, nxt_edge);
      load_flags(P.seg[c.seg], c.local(P) * SUB, nxt_mk);
    }
    while (c.live(P)) {
      uint4 v[GS];
      uint2 mk[GS];
#pragma unroll
      for (int j = 0; j < GS; j++) { v[j] = nxt[j]; mk[j] = nxt_mk[j]; }
      const uint32_t edge = nxt_edge;
      const uint32_t cur_macro = c.local(P);
      const bool last_group = g == GPM - 1;
      if (last_group) { c.unit += n_warps; c.settle_seg(P); g = 0; } else { g++; }
      if (c.live(P)) {
        load_group(P.seg[c.seg], c.local(P) * SUB + g * GS, nxt, nxt_edge);
        load_flags(P.seg[c.seg], c.local(P) * SUB + g * GS, nxt_mk);
      }
      filter_group(v, edge, mk);
      if (last_group) {
        W.consume_pending(acc);
        // same scoreboard trap as in the tile path: settle the prefetched group first
#pragma unroll
        for (int j = 0; j < GS; j++) {
          asm volatile("" : "+r"(nxt[j].x), "+r"(nxt[j].y), "+r"(nxt[j].z), "+r"(nxt[j].w));
          asm volatile("" : "+r"(nxt_mk[j].x), "+r"(nxt_mk[j].y));
        }
        asm volatile("" : "+r"(nxt_edge));
        const uint32_t w0[5] = {0, 0, 0, 0, 0};
        W.handle_hits(acc, 0, w0, cur_macro * SUB * WTILE);
        acc = 0;
        if (c.live(P) && c.seg != W.cur) {  // the warp's next unit lies in another stream
          W.drain();
          W.cur = c.seg;
        }
      }
    }
  } else {
  uint32_t nxt[5];
  if (c.live(P)) load_tile(P.seg[c.seg], c.local(P), lane, nxt);
  if constexpr (ScanWarp<D, NH, FM, PROF, RG>::LOCAL) {
    // Rotated loop: the table loads of tile t (its rounds) are issued at the top of
    // iteration t + 1, right after the prefetched words of tile t + 1 have been settled and
    // before tile t + 2 is requested; they are looked at after stage A of tile t + 1.  The
    // loop's back edge thus falls where no load is in flight (ptxas waits for the shared
    // scoreboard there).
    uint32_t w[5] = {0, 0, 0, 0, 0};
    uint32_t acc_prev = 0, base_prev = 0;
    while (c.live(P)) {
      W.settle(nxt);
      if (c.seg != W.cur) {  // first tile of another stream: finish the previous one's hits
        W.start_local(acc_prev, w, base_prev);
        W.drain();
        acc_prev = 0;
        W.cur = c.seg;
      }
      W.start_local(acc_prev, w, base_prev);
#pragma unroll
      for (int i = 0; i < 5; i++) w[i] = nxt[i];
      base_prev = c.local(P) * WTILE;
      c.unit += n_warps;
      c.settle_seg(P);
      if (c.live(P)) load_tile(P.seg[c.seg], c.local(P), lane, nxt);
      halo_finish(lane, w);
      uint32_t acc1;
      W.stage_a(w, acc_prev, acc1);
      W.resolve_local(acc_prev);
    }
    W.start_local(acc_prev, w, base_prev);  // the last tile's hits; drain() resolves them
  } else {
  while (c.live(P)) {
    uint32_t w[5];
#pragma unroll
    for (int i = 0; i < 5; i++) w[i] = nxt[i];
    const uint32_t tile_base = c.local(P) * WTILE;
    c.unit += n_warps;
    c.settle_seg(P);
    if (c.live(P)) load_tile(P.seg[c.seg], c.local(P), lane, nxt);
    halo_finish(lane, w);
    uint32_t acc0, acc1;
    W.stage_a(w, acc0, acc1);
    W.consume_pending(acc0 | acc1);
    W.settle(nxt);
    W.handle_hits(acc0, acc1, w, tile_base);
    if (c.live(P) && c.seg != W.cur) {  // the warp's next tile lies in another stream
      W.drain();
      W.cur = c.seg;
    }
  }
  }
  }
  W.drain();

  if (PROF) {
    unsigned long long v[4] = {W.n_bloom, W.n_seed, W.n_probe, W.n_hit};
#pragma unroll
    for (int i = 0; i < 4; i++) {
      unsigned long long s = v[i];
      for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(FULL_MASK, s, o);
      if (lane == 0 && s) atomicAdd(P.prof + i, s);
    }
  }
}

}  // namespace dkb

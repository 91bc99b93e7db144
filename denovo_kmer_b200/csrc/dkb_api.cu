// dkb_api.cu — the C ABI of include/dkb.h over the sm_100a kernels.
// No CPU fallback: every compute entry point needs a CUDA device.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "../../include/dkb.h"
#include "dkb_build.cuh"
#include "dkb_pack.cuh"
#include "dkb_regions.cuh"

using namespace dkb;
static_assert(DKB_MAX_MULTI == dkb::MAX_SEGMENTS, "ABI and kernel disagree on the batches per launch");

// A device buffer and its capacity, in elements.
template <typename T>
struct DevBuf {
  T *p = nullptr;
  size_t cap = 0;
  void free() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

// Page-locked host scratch and its capacity, in elements (grow_host).
template <typename T>
struct HostBuf {
  T *p = nullptr;
  size_t cap = 0;
  void free() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
};

struct dkb_ctx {
  int device = 0;
  int k = 0;
  int n_children = 1, n_samples = DKB_N_SAMPLES;  // a family: 2 + n_children samples
  int n_sms = 0;
  std::string err;

  dkb_tuning user_tuning{0, 0, 0, 0};
  int s = 0, D = 0, NH = 0;  // resolved at table build
  bool gf = false;           // seed filter probed in L2 instead of shared memory
  bool gate = false;         // stage A reads the flags and skips lookups of unusable seeds (modes 3, 4)
  uint32_t bloom_words = BLOOM_WORDS;

  // entries
  size_t n_entries = 0, n_live = 0;
  uint32_t n_variants = 0;
  uint64_t *d_keys = nullptr;
  uint32_t *d_variant = nullptr;
  uint8_t *d_allele = nullptr;
  uint8_t *d_dead = nullptr;
  // key table
  uint4 *d_tslots = nullptr;
  uint32_t table_slots = 0;
  // seeds
  uint4 *d_sslots = nullptr;  // seed table: 64-byte slots (seed + two records), 4 x uint4 each
  uint32_t *d_probe = nullptr;  // shared-memory filter mode: probe array in front of the slots
  uint32_t probe_slots = 0;
  bool canon = false;         // seeds keyed by their strand-canonical form
  uint32_t seed_slots = 0;
  uint32_t n_seeds = 0;
  uint32_t *d_bloom = nullptr, *d_pre = nullptr;
  uint32_t pre_words = 0;  // shared-memory pre-filter of the L2 filter mode
  bool want_pre = false;   // the tuner's choice
  uint64_t bloom_bits_set = 0;
  uint64_t occupied_halves = 0, direct_halves = 0;  // seed-record halves with a designation; direct ones
  // counters and results
  uint32_t *d_counts = nullptr;  // [n_samples][n_entries]
  uint32_t *d_hits = nullptr, *d_distinct = nullptr, *d_nkmers = nullptr;
  uint8_t *d_calls = nullptr;
  bool finalised = false;
  // inheritance (dkb_table_set_locus_classes, dkb_ctx_set_child_sexes): each variant's locus
  // class (null: all autosomal) and each child's sex
  uint8_t *d_cls = nullptr;  // [n_variants], allocated by the first dkb_table_set_locus_classes
  bool cls_on = false;       // d_cls holds classes in force (else: all autosomal)
  ChildSexes sexes = 0;
  // profiling counters
  bool prof = false;
  unsigned long long *d_prof = nullptr;
  // streams / staging for host batches
  cudaStream_t s_scan = nullptr, s_copy = nullptr;
  // per-launch CUDA-event timing of the scan kernel (pooled event pairs)
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pool, ev_pending;
  double scan_ms_total = 0.0;
  uint64_t scan_launches_timed = 0;
  float last_scan_ms = 0.f;
  // A staging slot: device buffers one launch's inputs are copied into.  Slots come in rings of
  // two, so that the copies for one launch overlap the scan of the previous one (stage_slot).
  struct Slot {
    cudaEvent_t copied = nullptr, freed = nullptr;  // on the copy / scan stream
    bool in_use = false;                            // a scan reads the slot until `freed`
    void free() {
      if (copied) cudaEventDestroy(copied);
      if (freed) cudaEventDestroy(freed);
      copied = freed = nullptr;
    }
  };
  template <typename S>
  struct Ring {
    S slot[2];
    int next = 0;
  };
  // host batches of every host submit form
  struct Stage : Slot {
    DevBuf<uint32_t> bases, mask;
    // raw reads for the device-side packer (dkb_batch_submit_reads and its multi form), each
    // array the batches' concatenated; the 4-bit form's nibble starts are computed into
    // nib_host and copied from there
    DevBuf<uint8_t> seq, qual;
    DevBuf<uint64_t> offsets, nib;
    HostBuf<uint64_t> nib_host;
    // zero lists of dkb_batch_submit_sparse and its multi form, concatenated
    DevBuf<uint32_t> zoff;
    DevBuf<uint8_t> zbytes;
    void free() {
      bases.free(); mask.free();
      seq.free(); qual.free(); offsets.free(); nib.free(); nib_host.free();
      zoff.free(); zbytes.free();
      Slot::free();
    }
  };
  Ring<Stage> stage;
  uint64_t scan_launches = 0, positions_scanned = 0;
  // multi-GPU: the communicator and the overlapped count reduction (dkb_reduce_push)
  void *comm = nullptr;  // ncclComm_t
  int rank = 0, world = 1;
  cudaStream_t s_side = nullptr;
  uint32_t *d_red[2] = {nullptr, nullptr};  // snapshots of the counters being summed
  size_t red_cap = 0;                       // capacity of each, in uint32
  cudaEvent_t ev_snap[2] = {nullptr, nullptr}, ev_red[2] = {nullptr, nullptr};
  int red_next = 0, red_pending = -1, red_last = -1;
  // the locus classes (copied, on the scan stream; null when all autosomal) and child sexes in
  // force when each snapshot was pushed: its kernel 3 uses these
  uint8_t *d_red_cls[2] = {nullptr, nullptr};
  bool red_has_cls[2] = {false, false};
  ChildSexes red_sexes[2] = {0, 0};
  // region mode (dkb_table_set_regions): each entry's variant window, and the loci the next
  // submit takes (host buffers, copied by that submit): one batch's (dkb_batch_set_loci) or
  // one set per batch of a multi-batch submit (dkb_batch_set_loci_multi)
  bool regions = false;
  ulonglong2 *d_entry_win = nullptr;
  struct Loci {
    const uint64_t *offsets = nullptr, *lo = nullptr, *hi = nullptr;
    size_t n_reads = 0;
    uint64_t n_pos = 0;
  } loci[DKB_MAX_MULTI];
  int loci_n = 0;           // batches the pending loci are for
  bool loci_set = false;    // loci are pending
  bool loci_multi = false;  // ... from dkb_batch_set_loci_multi
  // the read-locus index of one launch's batches on the device (concatenated, one segment per
  // batch with reads)
  struct LociStage : Slot {
    DevBuf<uint64_t> offsets, lo, hi;
    DevBuf<uint32_t> start, tile;
    DevBuf<ulonglong2> span;
    uint32_t tile_base[DKB_MAX_MULTI] = {}, n_tiles[DKB_MAX_MULTI] = {};  // per batch of the submit
    void free() {
      offsets.free(); lo.free(); hi.free();
      start.free(); tile.free(); span.free();
      Slot::free();
    }
  };
  Ring<LociStage> lstage;
};

namespace {

thread_local std::string g_err;

// Dynamic shared-memory limit and carve-out last set for each (device, scan kernel).  The
// attributes belong to the function, not to a context, and the size an L2-filter kernel needs
// changes with the pre-filter every table build chooses - so they are set again whenever the
// size differs from what the function was last given, by any context of this process.
std::mutex g_smem_mu;
std::map<std::pair<int, const void *>, size_t> g_smem_set;

int fail(dkb_ctx *ctx, int code, const std::string &msg) {
  if (ctx) ctx->err = msg;
  g_err = msg;
  return code;
}

#define CU(call)                                                                          \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess)                                                                \
      return fail(ctx, e_ == cudaErrorMemoryAllocation ? DKB_ENOMEM : DKB_ECUDA,          \
                  std::string(#call) + ": " + cudaGetErrorString(e_));                    \
  } while (0)

uint32_t pow2_at_least(uint64_t x) {
  uint32_t p = 1024;
  while (p < x && p < 0x80000000u) p <<= 1;
  return p;
}

template <typename T>
void dfree(T *&p) {
  if (p) cudaFree(p);
  p = nullptr;
}

// Forget whatever loci are pending, single-batch or multi-batch.
void drop_loci(dkb_ctx *c) { c->loci_set = false; }

void free_table(dkb_ctx *c) {
  dfree(c->d_keys); dfree(c->d_variant); dfree(c->d_allele); dfree(c->d_dead);
  dfree(c->d_tslots);
  dfree(c->d_sslots); dfree(c->d_probe); dfree(c->d_bloom); dfree(c->d_pre);
  c->probe_slots = 0;
  dfree(c->d_counts); dfree(c->d_hits);  // (d_distinct, d_nkmers live in d_hits' block)
  c->d_distinct = c->d_nkmers = nullptr;
  dfree(c->d_calls);
  dfree(c->d_entry_win);
  c->regions = false;  // a new table counts the whole stream until dkb_table_set_regions
  dfree(c->d_cls);
  c->cls_on = false;  // ... and is all autosomal until dkb_table_set_locus_classes
  for (int i = 0; i < 2; i++) dfree(c->d_red_cls[i]);
  drop_loci(c);
  c->n_entries = c->n_live = 0;
  c->occupied_halves = c->direct_halves = 0;
  c->n_variants = 0;
  c->finalised = false;
  c->red_pending = c->red_last = -1;  // snapshots of the old table's counters are void
}

// Words of the L2-resident seed filter: 64 bits per seed, between the shared-memory size
// and 32 MB (it shares L2 with the tables and the stream).
// Measured on the 100 000-candidate WGS shard (6 M seeds): 4 / 8 / 16 / 32 / 48 MB -> 2.89 / 3.65 /
// 3.86 / 3.92 / 3.91 Tbases/s: below 16 MB the filter's false positives (each a DRAM access
// into the 1.5 GB slot table) cost more than the filter's own L2 misses.
uint32_t l2_filter_words(double seeds) {
  const double cap = 8.0 * 1024 * 1024;  // 32 MB
  double w = seeds * 2.0;
  if (w > cap) w = cap;
  if (w < BLOOM_WORDS) w = BLOOM_WORDS;
  return (uint32_t)w;
}
// Shared-memory pre-filter of the L2 filter mode: 145 KB - with the 18 KB of lists and the
// 1 KB the system reserves it fills the 164 KB shared-memory carve-out exactly and leaves
// 92 KB of L1, whose lines track the outstanding L2 loads.  Measured on configs[1]
// (Tbases/s; profiles/README.md): 107 KB (132 KB carve-out) 4.64, 128 KB 4.91, 139 KB 5.04,
// 171 KB (196 KB carve-out, 60 KB of L1) 4.94, 192 KB 2.8.
constexpr uint32_t PRE_WORDS = 37120;

// Words of the pre-filter the build should use for this table (0 = none).  DKB_PREFILTER_WORDS overrides.
uint32_t pre_filter_words(bool want) {
  if (const char *e = getenv("DKB_PREFILTER_WORDS")) {
    long w = atol(e);
    if (w < 0) w = 0;
    if (w > BLOOM_WORDS) w = BLOOM_WORDS;
    return (uint32_t)(w / 4 * 4);
  }
  return want ? PRE_WORDS : 0;
}

// Ladder seeds one SNV-sized haplotype strand needs (k windows) at stride D, seed length s.
double ladder_seeds_per_strand(int k, int s, int D) {
  const int E = k - s, G = ((E + 1) / D) * D, nwin = k;
  double n = 0;
  for (int r = 0; r < D; r++) {
    const int base = E - ((E - r) % D);  // first ladder element of residue r
    n += 1 + (nwin - 1 > base ? (nwin - 1 - base + G - 1) / G : 0);
  }
  return n;
}

// Modelled cost of one 2048-position warp tile, in cycles per scheduler: filter lookups +
// handling of the filter's false positives + stage C for s-mers of unrelated sequence that
// equal a seed by chance.  Constants fitted to measured scan times (profiles/README.md):
//  * a shared-memory lookup ~16 cycles (bank-conflict wavefronts as much as its instructions);
//  * an L2 lookup 119: an SM sustains about one random L2 load per clock, shared by its four
//    schedulers and 32 lanes - but only while ~100 KB of L1 are left to track the loads;
//  * behind the 139 KB pre-filter an L2 lookup costs 22 + 105 x (fraction the pre-filter passes);
//  * a false positive 9 (strides <= 4: verified by its own lane) or 16 (macro tiles: compacted,
//    bases re-read from L2); a chance seed match 25 (one record compare);
//  * a seed table beyond L2 turns every probe into a DRAM access (factor `table`).
double tile_cost(double n_entries, bool hints, int k, int s, int D, int NH, bool gf, bool pre,
                 double *seeds_out) {
  const double n_haps = n_entries / k;  // allele haplotypes (SNV-sized)
  // both strands; ref/alt haplotypes share the seeds that avoid the variant base (x0.7)
  double seeds = n_haps * 2.0 * 0.7 * ladder_seeds_per_strand(k, s, D);
  if (!hints) seeds *= 2.3;  // min-hash rule: ~2/(w+1) density instead of 1/w
  if (canon_for_mode(gf ? 1 : 0)) seeds *= 0.5;  // both strands share their (canonical) seeds
  if (seeds_out) *seeds_out = seeds;
  const double bits = 32.0 * (gf ? l2_filter_words(seeds) : (double)BLOOM_WORDS);
  const double dens = 1.0 - exp(-NH * seeds / bits);
  const double fp = pow(dens, NH) * 1.3 + 1e-4;  // 1.3: per-word load variance
  const double lookups_lane = 64.0 / D, lookups_tile = 2048.0 / D;
  const double hits = lookups_tile * fp;
  const double chance = seeds / pow(4.0, s);  // P(random s-mer is a seed)
  const double table = seeds > 2e6 ? 3.0 : seeds > 5e5 ? 1.3 : 1.0;
  const double chance_cost = 25.0 * table * lookups_tile * chance;
  // (strides 8, 16: lookups gated by the flag stream cost ~8 more and reach the filter 0.58 times
  // as often at the usual 4 % of unusable positions; they are used when that pays - see the build)
  double l2_lookup = D >= 8 ? 8.0 + 0.58 * 119.0 : 119.0;
  if (pre) {
    const double pass = 1.0 - exp(-seeds / (32.0 * pre_filter_words(true)));
    l2_lookup = D >= 8 && pass > 0.55 ? 30.0 + 0.58 * 105.0 * pass : 22.0 + 105.0 * pass;
  }
  if (D >= 8)  // (round-2 refit: the probe array and normal-priority stream loads made the shared-memory mode cheaper)
    return (gf ? 61.0 : 37.0) + lookups_lane * (gf ? l2_lookup : 16.0 + NH) + (gf ? 16.0 : 14.6) * table * hits +
           chance_cost;
  return 100.0 + lookups_lane * (gf ? l2_lookup : 13.0 + 1.5 * NH) + 9.0 * table * (hits < 64 ? hits : 64) +
         (hits > 64 ? 14.0 * table * (hits - 64) : 0.0) + chance_cost;
}

// Resolve (s, D, NH): the caller's choice, else DKB_TUNING="s,D,NH", else the
// cheapest combination under tile_cost().
int resolve_tuning(dkb_ctx *ctx, size_t n_entries, bool hints) {
  dkb_tuning t = ctx->user_tuning;
  if (const char *e = getenv("DKB_TUNING")) {
    int a = 0, b = 0, c = 0, d = 0;
    if (sscanf(e, "%d,%d,%d,%d", &a, &b, &c, &d) >= 1) {
      if (!t.seed_len) t.seed_len = a;
      if (!t.stride) t.stride = b;
      if (!t.bloom_hashes) t.bloom_hashes = c;
      if (!t.filter_mode) t.filter_mode = d;
    }
  }
  const int k = ctx->k;
  if (t.stride != 0 && t.stride != 1 && t.stride != 2 && t.stride != 4 && t.stride != 8 &&
      t.stride != 16)
    return fail(ctx, DKB_EINVAL, "stride must be 1, 2, 4, 8 or 16");
  if (t.bloom_hashes < 0 || t.bloom_hashes > 4)
    return fail(ctx, DKB_EINVAL, "bloom_hashes must be 1..4");
  if (t.seed_len != 0 && (t.seed_len < 8 || t.seed_len > MAX_SEED_LEN))
    return fail(ctx, DKB_EINVAL, "seed_len out of range (8..15 and <= k - stride + 1)");
  if (t.filter_mode < 0 || t.filter_mode > 2)
    return fail(ctx, DKB_EINVAL, "filter_mode must be 0 (auto), 1 (shared memory) or 2 (L2)");
  int best_D = 0, best_NH = 0, best_s = 0, best_gf = 0;
  bool best_pre = false;
  double best = 1e300;
  for (int mode = 0; mode <= 2; mode++) {  // shared memory, L2, L2 behind the pre-filter
    const int gf = mode > 0;
    const bool pre = mode == 2;
    if (pre && pre_filter_words(true) == 0) continue;
    if (mode == 1 && getenv("DKB_PREFILTER_WORDS") && pre_filter_words(true) != 0) continue;
    if (t.filter_mode && t.filter_mode != gf + 1) continue;
    for (int D = 1; D <= 16; D *= 2) {
      if (t.stride && t.stride != D) continue;
      if (gf && D < 2) continue;  // the L2 mode is built for strides 2..16
      for (int s = 8; s <= MAX_SEED_LEN; s++) {
        if (t.seed_len && t.seed_len != s) continue;
        if (s > k - D + 1) continue;
        for (int NH = 1; NH <= 4; NH++) {
          if (gf && NH > 2) continue;
          if (t.bloom_hashes ? t.bloom_hashes != NH : NH > 2) continue;  // 3, 4: manual only
          const double c = tile_cost((double)n_entries, hints, k, s, D, NH, gf != 0, pre, nullptr);
          if (c < best) { best = c; best_D = D; best_NH = NH; best_s = s; best_gf = gf; best_pre = pre; }
        }
      }
    }
  }
  if (best_D == 0)
    return fail(ctx, DKB_EINVAL,
                "no (seed_len, stride, hashes, filter_mode) fits: need seed_len <= k - stride + 1; "
                "L2 mode takes strides 2..16 and 1..2 hashes");
  ctx->s = best_s;
  ctx->D = best_D;
  ctx->NH = best_NH;
  ctx->gf = best_gf != 0;
  ctx->want_pre = best_pre;
  return DKB_OK;
}

// Fold finished scan launches into the running totals; recycle their events.
void collect_timing(dkb_ctx *ctx) {
  size_t keep = 0;
  for (auto &pr : ctx->ev_pending) {
    float ms = 0.f;
    if (cudaEventQuery(pr.second) == cudaSuccess &&
        cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) {
      ctx->scan_ms_total += ms;
      ctx->scan_launches_timed++;
      ctx->last_scan_ms = ms;
      ctx->ev_pool.push_back(pr);
    } else {
      cudaGetLastError();
      ctx->ev_pending[keep++] = pr;
    }
  }
  ctx->ev_pending.resize(keep);
}

SeedTable seed_table(const dkb_ctx *ctx) {
  SeedTable T;
  T.slots = ctx->d_sslots;
  T.n_slots = ctx->seed_slots;
  T.probe = ctx->d_probe;
  T.n_probe = ctx->probe_slots;
  return T;
}

KeyTable key_table(const dkb_ctx *ctx) {
  KeyTable T;
  T.slots = ctx->d_tslots;
  T.bucket_mask = ctx->table_slots / KBUCKET - 1;
  return T;
}

typedef void (*scan_fn)(const ScanParams);
}  // namespace

// The scan kernel's instantiations are compiled one stride per translation unit
// (dkb_scan_inst.cu with -DDKB_INST_D=...), in parallel; each exports its picker.
namespace dkb {
scan_fn pick_scan_d1(int NH, int fm, bool prof, bool rg);
scan_fn pick_scan_d2(int NH, int fm, bool prof, bool rg);
scan_fn pick_scan_d4(int NH, int fm, bool prof, bool rg);
scan_fn pick_scan_d8(int NH, int fm, bool prof, bool rg);
scan_fn pick_scan_d16(int NH, int fm, bool prof, bool rg);
}  // namespace dkb

namespace {
scan_fn pick_scan(int D, int NH, int fm, bool prof, bool rg) {
  switch (D) {
    case 1: return pick_scan_d1(NH, fm, prof, rg);
    case 2: return pick_scan_d2(NH, fm, prof, rg);
    case 4: return pick_scan_d4(NH, fm, prof, rg);
    case 8: return pick_scan_d8(NH, fm, prof, rg);
    case 16: return pick_scan_d16(NH, fm, prof, rg);
  }
  return nullptr;
}

// The batches of one submit: batch i has n_positions[i] stream positions and is counted into
// the counters of samples[i].  Its packed streams are at d_bases[i] / d_mask[i] on the device:
// the caller's for the device forms, a staging slot's for the host forms (their staging step
// sets them).
struct Batches {
  bool multi;  // a multi-batch submit: it takes the loci of dkb_batch_set_loci_multi
  int n;
  const uint64_t *n_positions;
  const int *samples;
  const uint32_t *const *d_bases, *const *d_mask;
};

// One scan launch over the batches (each into its sample's counters).
// Region mode: ls is the read-locus index of all of them (stage_loci).
int launch_scan(dkb_ctx *ctx, const Batches &b, dkb_ctx::LociStage *ls) {
  const uint64_t *n_positions = b.n_positions;
  ScanParams P;
  memset(&P, 0, sizeof(P));
  // work units: tiles, or macro tiles of 4-8 tiles at strides 8/16
  const uint32_t per_unit = ctx->D >= 8 ? 32u / (64u / ctx->D) : 1u;
  uint64_t units = 0, total_pos = 0;
  P.n_seg = 0;
  for (int i = 0; i < b.n; i++) {
    if (n_positions[i] == 0) continue;
    ScanSegment &S = P.seg[P.n_seg++];
    S.bases = b.d_bases[i];
    S.mask = b.d_mask[i];
    S.counts = ctx->d_counts + (size_t)b.samples[i] * ctx->n_entries;
    S.n_pos = (uint32_t)n_positions[i];
    S.n_bwords = (uint32_t)dkb_stream_bases_words(n_positions[i]);
    S.n_mwords = (uint32_t)dkb_stream_mask_words(n_positions[i]);
    S.n_tiles = (uint32_t)((n_positions[i] + WTILE - 1) / WTILE);
    S.unit_begin = (uint32_t)units;
    units += (S.n_tiles + per_unit - 1) / per_unit;
    S.unit_end = (uint32_t)units;
    if (ls) {
      P.rseg[P.n_seg - 1].tile_base = ls->tile_base[i];
      P.rseg[P.n_seg - 1].n_tiles = ls->n_tiles[i];
    }
    total_pos += n_positions[i];
  }
  if (P.n_seg == 0) return DKB_OK;
  if (units >= 0xFFFF0000ull) return fail(ctx, DKB_EINVAL, "too many positions in one launch");
  for (int i = P.n_seg; i < MAX_SEGMENTS; i++) P.seg[i] = P.seg[P.n_seg - 1];  // never indexed; keep valid
  P.bloom = ctx->d_bloom;
  P.bloom_words = ctx->bloom_words;
  P.pre = ctx->d_pre;
  P.pre_words = ctx->gf ? ctx->pre_words : 0;
  P.st = seed_table(ctx);
  P.kt = key_table(ctx);
  P.seed_mult = SEED_MULT << (32 - 2 * ctx->s);
  P.seed_mask = (1u << (2 * ctx->s)) - 1;
  P.cshift = 32 - 2 * ctx->s;
  P.four = 4;
  for (int i = 0; i < 32; i++) P.pw[i] = 1u << i;
  P.filter_words = BLOOM_WORDS;
  P.k = ctx->k;
  P.s = ctx->s;
  P.prof = ctx->d_prof;
  const bool rg = ctx->regions;
  if (rg) {
    if (!ls) return fail(ctx, DKB_ESTATE, "region mode scans batches with their loci");
    P.read_start = ls->start.p;
    P.tile_read = ls->tile.p;
    P.read_span = ls->span.p;
    P.entry_win = ctx->d_entry_win;
  }
  scan_fn fn = pick_scan(ctx->D, ctx->NH, ctx->gf ? (ctx->pre_words ? 2 : 1) + (ctx->gate ? 2 : 0) : 0, ctx->prof, rg);
  if (!fn && rg && ctx->prof)
    return fail(ctx, DKB_ESTATE, "region mode has no scan kernel with profiling counters (dkb_profile_counters 0)");
  if (!fn) return fail(ctx, DKB_EINVAL, "no scan kernel for this tuning");
  size_t smem_bytes = !ctx->gf ? SCAN_SMEM_BYTES
                      : ctx->pre_words ? SCAN_SMEM_BYTES_PRE + (size_t)ctx->pre_words * 4 : SCAN_SMEM_BYTES_GF;
  {
    std::lock_guard<std::mutex> lk(g_smem_mu);
    auto it = g_smem_set.find({ctx->device, (const void *)fn});
    if (it == g_smem_set.end() || it->second != smem_bytes) {
      CU(cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)smem_bytes));
      // L2 filter mode: as much L1 as the block leaves - the smallest carve-out that holds it
      // (+ 1 KB the system reserves); the hint is a percentage of 228 KB that the driver rounds
      // UP to a supported size.  Shared-memory filter mode: everything.
      CU(cudaFuncSetAttribute((const void *)fn, cudaFuncAttributePreferredSharedMemoryCarveout,
                              ctx->gf ? (int)(100 * (smem_bytes + 1024) / (228 * 1024))
                                      : (int)cudaSharedmemCarveoutMaxShared));
      g_smem_set[{ctx->device, (const void *)fn}] = smem_bytes;
    }
  }
  // one CTA per SM; short batches get one CTA per work unit so that they still spread over the SMs
  uint32_t grid = (uint32_t)units;
  if (grid > (uint32_t)ctx->n_sms) grid = ctx->n_sms;
  if (ctx->ev_pending.size() >= 256) collect_timing(ctx);
  std::pair<cudaEvent_t, cudaEvent_t> ev{nullptr, nullptr};
  if (!ctx->ev_pool.empty()) {
    ev = ctx->ev_pool.back();
    ctx->ev_pool.pop_back();
  } else {
    CU(cudaEventCreate(&ev.first));
    CU(cudaEventCreate(&ev.second));
  }
  CU(cudaEventRecord(ev.first, ctx->s_scan));
  fn<<<grid, SCAN_THREADS, smem_bytes, ctx->s_scan>>>(P);
  CU(cudaGetLastError());
  CU(cudaEventRecord(ev.second, ctx->s_scan));
  ctx->ev_pending.push_back(ev);
  ctx->scan_launches++;
  ctx->positions_scanned += total_pos;
  ctx->finalised = false;
  return DKB_OK;
}

// The slot protocol of both staging rings.  stage_slot takes the ring's next slot; fill(slot)
// grows its buffers (grow) and queues the copies of one launch's inputs into them on the copy
// stream, which first waits until the slot's last scan is done with them; the scan stream then
// waits for the copies.  release() hands the slots of a launch back once its scan is queued.
template <typename S, typename Fill>
int stage_slot(dkb_ctx *ctx, dkb_ctx::Ring<S> &ring, S *&out, Fill fill) {
  S &st = ring.slot[ring.next];
  ring.next ^= 1;
  if (st.in_use) CU(cudaStreamWaitEvent(ctx->s_copy, st.freed, 0));
  int rc = fill(st);
  if (rc != DKB_OK) return rc;
  CU(cudaEventRecord(st.copied, ctx->s_copy));
  CU(cudaStreamWaitEvent(ctx->s_scan, st.copied, 0));
  out = &st;
  return DKB_OK;
}

// Grow a buffer of slot st to at least `need` elements.  The slot's last scan may still read
// the old buffer, so the host waits for that scan first - only when the buffer must grow.
template <typename T>
int grow(dkb_ctx *ctx, dkb_ctx::Slot &st, DevBuf<T> &b, size_t need) {
  if (b.cap >= need) return DKB_OK;
  if (st.in_use) CU(cudaEventSynchronize(st.freed));
  b.free();  // a failed allocation must not leave a capacity behind a null pointer
  const size_t want = need + need / 8 + 256;
  T *q = nullptr;
  CU(cudaMalloc(&q, want * sizeof(T)));
  b.p = q;
  b.cap = want;
  return DKB_OK;
}

int release(dkb_ctx *ctx, std::initializer_list<dkb_ctx::Slot *> slots) {
  for (dkb_ctx::Slot *st : slots) {
    if (!st) continue;
    CU(cudaEventRecord(st->freed, ctx->s_scan));
    st->in_use = true;
  }
  return DKB_OK;
}

// Grow a slot's page-locked host scratch to at least `need` elements.  The caller has waited
// for the slot's last copies (its `copied` event): they may still read the old scratch.
template <typename T>
int grow_host(dkb_ctx *ctx, HostBuf<T> &b, size_t need) {
  if (b.cap >= need) return DKB_OK;
  b.free();
  const size_t want = need + need / 8 + 256;
  T *q = nullptr;
  CU(cudaMallocHost(&q, want * sizeof(T)));
  b.p = q;
  b.cap = want;
  return DKB_OK;
}

// Where a submit's packed streams go in a staging slot: batch i's at bases.p + bo[i] and
// mask.p + mo[i], each at a 16-byte-aligned offset; bw / mw words in all.
struct StreamLayout {
  size_t bo[DKB_MAX_MULTI], mo[DKB_MAX_MULTI], bw = 0, mw = 0;
  explicit StreamLayout(const Batches &b) {
    for (int i = 0; i < b.n; i++) {
      bo[i] = bw;
      mo[i] = mw;
      bw += (dkb_stream_bases_words(b.n_positions[i]) + 3) / 4 * 4;
      mw += (dkb_stream_mask_words(b.n_positions[i]) + 3) / 4 * 4;
    }
  }
  // grow the slot's stream buffers to hold the layout
  int grow_slot(dkb_ctx *ctx, dkb_ctx::Stage &st) const {
    int rc;
    if ((rc = grow(ctx, st, st.bases, bw)) != DKB_OK) return rc;
    return grow(ctx, st, st.mask, mw);
  }
  // the batches' device addresses, for launch_scan
  void place(const Batches &b, const dkb_ctx::Stage &st, const uint32_t **d_bases, const uint32_t **d_mask) const {
    for (int i = 0; i < b.n; i++) {
      d_bases[i] = st.bases.p + bo[i];
      d_mask[i] = st.mask.p + mo[i];
    }
  }
};

// Copy n host-resident batches into one staging buffer (StreamLayout).  d_bases / d_mask get
// the batches' device addresses.
int stage_batches(dkb_ctx *ctx, const Batches &b, const uint32_t *const *bases2, const uint32_t *const *mask1,
                  const uint32_t **d_bases, const uint32_t **d_mask, dkb_ctx::Stage *&out) {
  const uint64_t *n_positions = b.n_positions;
  const StreamLayout L(b);
  return stage_slot(ctx, ctx->stage, out, [&](dkb_ctx::Stage &st) -> int {
    int rc;
    if ((rc = L.grow_slot(ctx, st)) != DKB_OK) return rc;
    L.place(b, st, d_bases, d_mask);
    for (int i = 0; i < b.n; i++) {
      if (n_positions[i] == 0) continue;
      CU(cudaMemcpyAsync(st.bases.p + L.bo[i], bases2[i], dkb_stream_bases_words(n_positions[i]) * 4,
                         cudaMemcpyHostToDevice, ctx->s_copy));
      CU(cudaMemcpyAsync(st.mask.p + L.mo[i], mask1[i], dkb_stream_mask_words(n_positions[i]) * 4,
                         cudaMemcpyHostToDevice, ctx->s_copy));
    }
    return DKB_OK;
  });
}

// "batch i: " in front of a refusal that concerns one batch of a multi-batch submit
std::string batch_prefix(const Batches &b, int i) {
  return b.multi ? "batch " + std::to_string(i) + ": " : std::string();
}

// Host batches with their flags as zero lists: the bases and the zero lists are copied into
// one staging slot, concatenated, and ONE k_expand_zero_list launch writes every batch's flags
// into the slot's stream buffer (StreamLayout) ahead of the scan.
int stage_sparse(dkb_ctx *ctx, const Batches &b, const uint32_t *const *bases2, const uint32_t *const *zoff,
                 const uint8_t *const *zbytes, const size_t *zbytes_used, const uint32_t **d_bases,
                 const uint32_t **d_mask, dkb_ctx::Stage *&slot) {
  // the zero lists are checked here, once the batches' lengths are: their sizes follow from n_positions
  size_t nb[DKB_MAX_MULTI], zo[DKB_MAX_MULTI], zbo[DKB_MAX_MULTI], n_zoff = 0, n_zbytes = 0;
  for (int i = 0; i < b.n; i++) {
    nb[i] = dkb_zero_list_blocks(b.n_positions[i]);
    zo[i] = n_zoff;
    zbo[i] = n_zbytes;
    if (b.n_positions[i] == 0) continue;
    const uint32_t *z = zoff[i];
    if ((z[nb[i]] & 0x7FFFFFFFu) != zbytes_used[i])
      return fail(ctx, DKB_EINVAL, batch_prefix(b, i) + "zoff[n_blocks] != zbytes_used");
    // the expander trusts the offsets: they must ascend inside zbytes, a plain-bits block is 256 bytes
    for (size_t j = 0; j < nb[i]; j++) {
      const uint32_t cur = z[j] & 0x7FFFFFFFu, nxt = z[j + 1] & 0x7FFFFFFFu;
      if (nxt < cur || nxt > zbytes_used[i] || ((z[j] & 0x80000000u) && nxt - cur != 256u))
        return fail(ctx, DKB_EINVAL, batch_prefix(b, i) + "malformed zero list (block offsets)");
    }
    n_zoff += nb[i] + 1;
    n_zbytes += zbytes_used[i];
  }
  const StreamLayout L(b);
  int rc = stage_slot(ctx, ctx->stage, slot, [&](dkb_ctx::Stage &st) -> int {
    int rc;
    if ((rc = L.grow_slot(ctx, st)) != DKB_OK) return rc;
    if ((rc = grow(ctx, st, st.zoff, n_zoff)) != DKB_OK) return rc;
    if ((rc = grow(ctx, st, st.zbytes, n_zbytes ? n_zbytes : 1)) != DKB_OK) return rc;
    for (int i = 0; i < b.n; i++) {
      if (b.n_positions[i] == 0) continue;
      CU(cudaMemcpyAsync(st.bases.p + L.bo[i], bases2[i], dkb_stream_bases_words(b.n_positions[i]) * 4,
                         cudaMemcpyHostToDevice, ctx->s_copy));
      CU(cudaMemcpyAsync(st.zoff.p + zo[i], zoff[i], (nb[i] + 1) * 4, cudaMemcpyHostToDevice, ctx->s_copy));
      if (zbytes_used[i])
        CU(cudaMemcpyAsync(st.zbytes.p + zbo[i], zbytes[i], zbytes_used[i], cudaMemcpyHostToDevice, ctx->s_copy));
    }
    return DKB_OK;
  });
  if (rc != DKB_OK) return rc;
  ZeroListParams Z;
  memset(&Z, 0, sizeof(Z));
  for (int i = 0; i < b.n; i++) {
    if (b.n_positions[i] == 0) continue;
    ZeroListSegment &S = Z.seg[Z.n_seg++];
    S.zoff = slot->zoff.p + zo[i];
    S.zbytes = slot->zbytes.p + zbo[i];
    S.mask1 = slot->mask.p + L.mo[i];
    S.b_begin = Z.n_blocks;
    S.n_blocks = (uint32_t)nb[i];
    S.n_mwords = (uint32_t)dkb_stream_mask_words(b.n_positions[i]);
    Z.n_blocks += (uint32_t)nb[i];
  }
  k_expand_zero_list<<<(Z.n_blocks + 7) / 8, 256, 0, ctx->s_scan>>>(Z);
  CU(cudaGetLastError());
  L.place(b, *slot, d_bases, d_mask);
  return DKB_OK;
}

// Host batches of decoded reads: their bases, qualities and offsets are copied into one staging
// slot, concatenated, and ONE k_pack launch packs every batch into the slot's stream buffer
// (StreamLayout) ahead of the scan.  seq[i] points at batch i's first 4-bit byte (seq_format 1)
// or at the base its offsets count from (0); qual (may be null) and qual[i] (may be null) alike.
int stage_reads(dkb_ctx *ctx, const Batches &b, const uint8_t *const *seq, int seq_format,
                const uint8_t *const *qual, const uint64_t *const *offsets, const size_t *n_reads,
                int min_baseq, const uint32_t **d_bases, const uint32_t **d_mask, dkb_ctx::Stage *&slot) {
  const bool four_bit = seq_format == 1;
  // per batch with positions: its bases and where its seq / qual / offsets / nibble starts go
  uint64_t n_bases[DKB_MAX_MULTI], seq_bytes[DKB_MAX_MULTI];
  size_t so[DKB_MAX_MULTI], qo[DKB_MAX_MULTI], oo[DKB_MAX_MULTI], no[DKB_MAX_MULTI];
  size_t n_seq = 0, n_qual = 0, n_off = 0, n_nib = 0;
  for (int i = 0; i < b.n; i++) {
    so[i] = n_seq; qo[i] = n_qual; oo[i] = n_off; no[i] = n_nib;
    if (b.n_positions[i] == 0) continue;
    n_bases[i] = offsets[i][n_reads[i]] - offsets[i][0];
    seq_bytes[i] = n_bases[i];
    if (four_bit) {  // BAM keeps every read's 4-bit codes byte-aligned: (len + 1) / 2 bytes per read
      seq_bytes[i] = 0;
      for (size_t r = 0; r < n_reads[i]; r++) seq_bytes[i] += (offsets[i][r + 1] - offsets[i][r] + 1) / 2;
      n_nib += n_reads[i];
    }
    n_seq += seq_bytes[i];
    if (qual && qual[i]) n_qual += n_bases[i];
    n_off += n_reads[i] + 1;
  }
  const StreamLayout L(b);
  int rc = stage_slot(ctx, ctx->stage, slot, [&](dkb_ctx::Stage &st) -> int {
    int rc;
    if ((rc = L.grow_slot(ctx, st)) != DKB_OK) return rc;
    if ((rc = grow(ctx, st, st.seq, n_seq ? n_seq : 1)) != DKB_OK) return rc;
    if (n_qual && (rc = grow(ctx, st, st.qual, n_qual)) != DKB_OK) return rc;
    if ((rc = grow(ctx, st, st.offsets, n_off)) != DKB_OK) return rc;
    if (four_bit) {
      if ((rc = grow(ctx, st, st.nib, n_nib)) != DKB_OK) return rc;
      // the nibble starts go through the slot's page-locked scratch, which the slot's last
      // copies may still read: wait for those copies (not for any scan) before rewriting it
      CU(cudaEventSynchronize(st.copied));
      if ((rc = grow_host(ctx, st.nib_host, n_nib)) != DKB_OK) return rc;
    }
    for (int i = 0; i < b.n; i++) {
      if (b.n_positions[i] == 0) continue;
      const uint64_t *off = offsets[i];
      // the reads of a batch start at off[0] in the caller's arrays; device copies start at the batch's segment
      CU(cudaMemcpyAsync(st.seq.p + so[i], four_bit ? seq[i] : seq[i] + off[0], seq_bytes[i], cudaMemcpyHostToDevice,
                         ctx->s_copy));
      if (qual && qual[i])
        CU(cudaMemcpyAsync(st.qual.p + qo[i], qual[i] + off[0], n_bases[i], cudaMemcpyHostToDevice, ctx->s_copy));
      CU(cudaMemcpyAsync(st.offsets.p + oo[i], off, (n_reads[i] + 1) * 8, cudaMemcpyHostToDevice, ctx->s_copy));
      if (four_bit) {
        uint64_t *nib = st.nib_host.p + no[i], bytes = 0;
        for (size_t r = 0; r < n_reads[i]; r++) {
          nib[r] = bytes;
          bytes += (off[r + 1] - off[r] + 1) / 2;
        }
        CU(cudaMemcpyAsync(st.nib.p + no[i], nib, n_reads[i] * 8, cudaMemcpyHostToDevice, ctx->s_copy));
      }
    }
    return DKB_OK;
  });
  if (rc != DKB_OK) return rc;
  PackParams Q;
  memset(&Q, 0, sizeof(Q));
  for (int i = 0; i < b.n; i++) {
    if (b.n_positions[i] == 0) continue;
    PackSegment &S = Q.seg[Q.n_seg++];
    S.seq = slot->seq.p + so[i];
    S.qual = qual && qual[i] ? slot->qual.p + qo[i] : nullptr;
    S.offsets = slot->offsets.p + oo[i];
    S.nib_start = four_bit ? slot->nib.p + no[i] : nullptr;
    S.bases2 = slot->bases.p + L.bo[i];
    S.mask1 = slot->mask.p + L.mo[i];
    S.m_begin = Q.n_mwords;
    S.n_pos = b.n_positions[i];
    S.n_reads = (uint32_t)n_reads[i];
    S.n_bwords = (uint32_t)dkb_stream_bases_words(b.n_positions[i]);
    S.n_mwords = (uint32_t)dkb_stream_mask_words(b.n_positions[i]);
    Q.n_mwords += S.n_mwords;
  }
  Q.min_baseq = min_baseq;
  Q.four_bit = seq_format;
  const int TB = 256;
  k_pack<<<(uint32_t)((Q.n_mwords + TB - 1) / TB), TB, 0, ctx->s_scan>>>(Q);
  CU(cudaGetLastError());
  L.place(b, *slot, d_bases, d_mask);
  return DKB_OK;
}

const char *const NO_PROF_REGIONS = "region mode has no scan kernel with profiling counters (dkb_profile_counters 0)";

// Region mode: take the loci pending for this submit, whatever its outcome - dkb_batch_set_loci's
// for a single-batch submit, dkb_batch_set_loci_multi's for a multi-batch one - into l[0, n).
int take_loci(dkb_ctx *ctx, bool multi, dkb_ctx::Loci *l, int &n) {
  const bool set = ctx->loci_set;
  n = ctx->loci_n;
  for (int i = 0; i < n; i++) l[i] = ctx->loci[i];
  drop_loci(ctx);
  if (set && ctx->loci_multi != multi)
    return fail(ctx, DKB_ESTATE, multi ? "region mode: single-batch loci are pending, but this is a multi-batch submit"
                                       : "region mode: multi-batch loci are pending, but this is a single-batch submit");
  if (!set)
    return fail(ctx, DKB_ESTATE, multi ? "region mode: dkb_batch_set_loci_multi must come before every multi-batch submit"
                                       : "region mode: dkb_batch_set_loci must come before every single-batch submit");
  if (ctx->prof) return fail(ctx, DKB_ESTATE, NO_PROF_REGIONS);
  return DKB_OK;
}

// Region mode: the taken loci must be for the submit's batches and cover their positions.
int check_loci_positions(dkb_ctx *ctx, const Batches &b, const dkb_ctx::Loci *l, int n) {
  if (n != b.n)
    return fail(ctx, DKB_EINVAL, "the loci are for " + std::to_string(n) + " batches, the submit has " +
                                     std::to_string(b.n));
  for (int i = 0; i < n; i++)
    if (l[i].n_pos != b.n_positions[i])
      return fail(ctx, DKB_EINVAL, batch_prefix(b, i) + "the loci's reads cover " + std::to_string(l[i].n_pos) +
                                       " stream positions, the batch " + std::to_string(b.n_positions[i]));
  return DKB_OK;
}

// Copy the loci of a launch's n batches (copy stream) into one LociStage, concatenated, and
// build their read-locus index with one launch of each index kernel (scan stream, ahead of the
// scan).  ls = nullptr when no batch has reads (nothing to scan).
int stage_loci(dkb_ctx *ctx, int n, const dkb_ctx::Loci *l, dkb_ctx::LociStage *&ls) {
  ls = nullptr;
  LociSegments S;
  memset(&S, 0, sizeof(S));
  uint32_t tile_base[DKB_MAX_MULTI], n_tiles[DKB_MAX_MULTI];
  int batch_of[DKB_MAX_MULTI];
  size_t nr = 0, nt = 0;
  for (int i = 0; i < n; i++) {
    tile_base[i] = (uint32_t)nt;
    n_tiles[i] = 0;
    if (l[i].n_reads == 0) continue;  // (no positions: launch_scan skips the batch too)
    n_tiles[i] = (uint32_t)((l[i].n_pos + (1u << LOCI_TILE_SHIFT) - 1) >> LOCI_TILE_SHIFT);
    S.read_base[S.n_seg] = (uint32_t)nr;
    S.tile_base[S.n_seg] = (uint32_t)nt;
    batch_of[S.n_seg++] = i;
    nr += l[i].n_reads;
    nt += n_tiles[i] + 1;
  }
  if (S.n_seg == 0) return DKB_OK;
  S.read_base[S.n_seg] = (uint32_t)nr;
  S.tile_base[S.n_seg] = (uint32_t)nt;
  const size_t no = nr + S.n_seg;  // offsets: n_reads + 1 per segment
  int rc = stage_slot(ctx, ctx->lstage, ls, [&](dkb_ctx::LociStage &st) -> int {
    int rc;
    if ((rc = grow(ctx, st, st.offsets, no)) != DKB_OK) return rc;
    if ((rc = grow(ctx, st, st.lo, nr)) != DKB_OK) return rc;
    if ((rc = grow(ctx, st, st.hi, nr)) != DKB_OK) return rc;
    if ((rc = grow(ctx, st, st.start, nr)) != DKB_OK) return rc;
    if ((rc = grow(ctx, st, st.span, nr)) != DKB_OK) return rc;
    if ((rc = grow(ctx, st, st.tile, nt)) != DKB_OK) return rc;
    for (uint32_t j = 0; j < S.n_seg; j++) {
      const dkb_ctx::Loci &b = l[batch_of[j]];
      const size_t r0 = S.read_base[j];
      CU(cudaMemcpyAsync(st.offsets.p + r0 + j, b.offsets, (b.n_reads + 1) * 8, cudaMemcpyHostToDevice, ctx->s_copy));
      CU(cudaMemcpyAsync(st.lo.p + r0, b.lo, b.n_reads * 8, cudaMemcpyHostToDevice, ctx->s_copy));
      CU(cudaMemcpyAsync(st.hi.p + r0, b.hi, b.n_reads * 8, cudaMemcpyHostToDevice, ctx->s_copy));
    }
    return DKB_OK;
  });
  if (rc != DKB_OK) return rc;
  const int TB = 256;
  k_read_loci<<<(uint32_t)((nr + TB - 1) / TB), TB, 0, ctx->s_scan>>>(S, ls->offsets.p, ls->lo.p, ls->hi.p,
                                                                     ls->start.p, ls->span.p);
  k_tile_reads<<<(uint32_t)((nt + TB - 1) / TB), TB, 0, ctx->s_scan>>>(S, ls->start.p, ls->tile.p);
  CU(cudaGetLastError());
  for (int i = 0; i < n; i++) {
    ls->tile_base[i] = tile_base[i];
    ls->n_tiles[i] = n_tiles[i];
  }
  return DKB_OK;
}

// ---- host memory next to the GPU ---------------------------------------------------------
// NUMA node of the device's PCIe slot (-1 if the system does not say) and that node's CPUs.
int gpu_numa_node(int device) {
  char bus[32] = {0};
  if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) {
    cudaGetLastError();
    return -1;
  }
  for (char *c = bus; *c; c++) *c = (char)tolower(*c);
  std::ifstream f(std::string("/sys/bus/pci/devices/") + bus + "/numa_node");
  int node = -1;
  if (!(f >> node)) return -1;
  return node;
}

bool node_cpus(int node, cpu_set_t *set) {
  std::ifstream f("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist");
  std::string list;
  if (!std::getline(f, list)) return false;
  CPU_ZERO(set);
  int n = 0;
  size_t i = 0;
  while (i < list.size()) {  // "0-31,64-95"
    char *end = nullptr;
    long a = strtol(list.c_str() + i, &end, 10), b = a;
    if (end == list.c_str() + i) break;
    i = end - list.c_str();
    if (i < list.size() && list[i] == '-') {
      b = strtol(list.c_str() + i + 1, &end, 10);
      i = end - list.c_str();
    }
    for (long c = a; c <= b && c < CPU_SETSIZE; c++) { CPU_SET((int)c, set); n++; }
    if (i < list.size() && list[i] == ',') i++;
  }
  return n > 0;
}

// Prefer `node` for this thread's page allocations (-1: back to the default policy).  Best
// effort: containers often forbid the call, and then CPU affinity + first touch decide.
void prefer_node(int node) {
#ifdef SYS_set_mempolicy
  if (node < 0) {
    syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0);
    return;
  }
  unsigned long mask[16] = {0};
  if (node >= (int)(sizeof(mask) * 8)) return;
  mask[node / (8 * sizeof(long))] |= 1ul << (node % (8 * sizeof(long)));
  syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, sizeof(mask) * 8);
#else
  (void)node;
#endif
}

// ---- NCCL, bound at run time ---------------------------------------------------------
// libnccl.so.2 is opened with dlopen the first time a communicator is asked for, so a
// single-GPU user needs no NCCL at all; in a process that already holds NCCL (PyTorch's
// bundled copy) the same library instance is used.  Only the calls below are needed; their
// C signatures are stable across NCCL 2.x.
struct NcclId { char internal[128]; };  // ncclUniqueId
struct Nccl {
  void *h = nullptr;
  int (*GetUniqueId)(NcclId *) = nullptr;
  int (*CommInitRank)(void **, int, NcclId, int) = nullptr;
  int (*CommDestroy)(void *) = nullptr;
  int (*CommCount)(void *, int *) = nullptr;
  int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
  int (*GetVersion)(int *) = nullptr;
  std::string err;
};
constexpr int NCCL_UINT32 = 3, NCCL_SUM = 0;  // ncclUint32, ncclSum

Nccl *nccl() {
  static Nccl N;
  static std::once_flag once;
  std::call_once(once, [] {
    const char *names[] = {getenv("DKB_NCCL_LIBRARY"), "libnccl.so.2", "libnccl.so"};
    for (const char *nm : names) {
      if (!nm || !*nm) continue;
      if ((N.h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL))) break;
      N.err = dlerror();
    }
    if (!N.h) return;
    auto sym = [&](const char *name) {
      void *p = dlsym(N.h, name);
      if (!p) N.err = std::string("missing NCCL symbol ") + name;
      return p;
    };
    N.GetUniqueId = (decltype(N.GetUniqueId))sym("ncclGetUniqueId");
    N.CommInitRank = (decltype(N.CommInitRank))sym("ncclCommInitRank");
    N.CommDestroy = (decltype(N.CommDestroy))sym("ncclCommDestroy");
    N.CommCount = (decltype(N.CommCount))sym("ncclCommCount");
    N.AllReduce = (decltype(N.AllReduce))sym("ncclAllReduce");
    N.GetErrorString = (decltype(N.GetErrorString))sym("ncclGetErrorString");
    N.GetVersion = (decltype(N.GetVersion))sym("ncclGetVersion");
    if (!N.GetUniqueId || !N.CommInitRank || !N.CommDestroy || !N.AllReduce || !N.GetErrorString) {
      dlclose(N.h);
      N.h = nullptr;
    }
  });
  return &N;
}

#define NC(call)                                                                              \
  do {                                                                                        \
    int r_ = (call);                                                                          \
    if (r_ != 0)                                                                              \
      return fail(ctx, DKB_ENCCL, std::string(#call) + ": " + nccl()->GetErrorString(r_));    \
  } while (0)

// Side stream, events and the two snapshot buffers of the overlapped reduction.
int reduce_setup(dkb_ctx *ctx) {
  const size_t need = (ctx->n_entries ? ctx->n_entries : 1) * ctx->n_samples;
  if (!ctx->s_side) {
    CU(cudaStreamCreateWithFlags(&ctx->s_side, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
      CU(cudaEventCreateWithFlags(&ctx->ev_snap[i], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&ctx->ev_red[i], cudaEventDisableTiming));
    }
  }
  if (ctx->red_cap < need) {
    CU(cudaStreamSynchronize(ctx->s_side));
    CU(cudaStreamSynchronize(ctx->s_scan));
    for (int i = 0; i < 2; i++) dfree(ctx->d_red[i]);
    ctx->red_cap = 0;
    for (int i = 0; i < 2; i++) CU(cudaMalloc(&ctx->d_red[i], need * 4));
    ctx->red_cap = need;
    ctx->red_pending = ctx->red_last = -1;
  }
  return DKB_OK;
}

int finalise_counts(dkb_ctx *ctx, const dkb_thresholds *thr, const uint32_t *d_counts, const uint8_t *cls,
                    const ChildSexes &sexes);

// Samples a submit may name: [0, n_samples).
int check_sample(dkb_ctx *ctx, int sample) {
  if (sample >= 0 && sample < ctx->n_samples) return DKB_OK;
  return fail(ctx, DKB_EINVAL, ctx->n_samples == DKB_N_SAMPLES
                                   ? std::string("sample must be 0, 1 or 2")
                                   : "sample must be in [0, " + std::to_string(ctx->n_samples) + ")");
}

// The checks of the packed-stream forms (dkb_batch_submit, _device and their multi forms):
// n_batches and the arrays of a multi-batch submit, then the stream pointers of every batch
// with positions, which on the device must be aligned too.
int check_streams(dkb_ctx *ctx, const Batches &b, const uint32_t *const *bases2, const uint32_t *const *mask1,
                  bool device) {
  if (b.multi && (b.n < 0 || b.n > DKB_MAX_MULTI)) return fail(ctx, DKB_EINVAL, "n_batches out of range");
  if (b.multi && b.n && (!bases2 || !mask1 || !b.n_positions || !b.samples))
    return fail(ctx, DKB_EINVAL, "null argument");
  for (int i = 0; i < b.n; i++) {
    if (b.n_positions[i] == 0) continue;
    if (!bases2[i] || !mask1[i]) return fail(ctx, DKB_EINVAL, "null stream pointer");
    if (device && ((uintptr_t)bases2[i] & 15)) return fail(ctx, DKB_EINVAL, "d_bases2 must be 16-byte aligned");
    if (device && ((uintptr_t)mask1[i] & 3)) return fail(ctx, DKB_EINVAL, "d_mask1 must be 4-byte aligned");
  }
  return DKB_OK;
}

// The checks of the zero-list forms (dkb_batch_submit_sparse and its multi form); the zero
// lists themselves are checked by stage_sparse.
int check_sparse(dkb_ctx *ctx, const Batches &b, const uint32_t *const *bases2, const uint32_t *const *zoff,
                 const uint8_t *const *zbytes, const size_t *zbytes_used) {
  if (b.multi && (b.n < 0 || b.n > DKB_MAX_MULTI)) return fail(ctx, DKB_EINVAL, "n_batches out of range");
  if (b.multi && b.n && (!bases2 || !zoff || !zbytes || !zbytes_used || !b.n_positions || !b.samples))
    return fail(ctx, DKB_EINVAL, "null argument");
  for (int i = 0; i < b.n; i++)
    if (b.n_positions[i] && (!bases2[i] || !zoff[i] || (zbytes_used[i] && !zbytes[i])))
      return fail(ctx, DKB_EINVAL, batch_prefix(b, i) + "null stream pointer");
  return DKB_OK;
}

// The checks of the decoded-read forms (dkb_batch_submit_reads and its multi form).  Sets each
// batch's stream positions, n_pos[i] (0 for a batch without reads).
int check_reads(dkb_ctx *ctx, const Batches &b, const uint8_t *const *seq, int seq_format,
                const uint64_t *const *offsets, const size_t *n_reads, uint64_t *n_pos) {
  if (b.multi && (b.n < 0 || b.n > DKB_MAX_MULTI)) return fail(ctx, DKB_EINVAL, "n_batches out of range");
  if (seq_format != 0 && seq_format != 1) return fail(ctx, DKB_EINVAL, "seq_format must be 0 (ASCII) or 1 (BAM 4-bit)");
  if (b.multi && b.n && (!seq || !offsets || !n_reads || !b.samples)) return fail(ctx, DKB_EINVAL, "null argument");
  for (int i = 0; i < b.n; i++) {
    if (n_reads[i] == 0) continue;
    if (!seq[i] || !offsets[i]) return fail(ctx, DKB_EINVAL, batch_prefix(b, i) + "null read buffer");
    if (n_reads[i] >= 0xFFFFFFFFull) return fail(ctx, DKB_EINVAL, batch_prefix(b, i) + "too many reads in one batch");
    for (size_t r = 0; r < n_reads[i]; r++)
      if (offsets[i][r + 1] < offsets[i][r])
        return fail(ctx, DKB_EINVAL, batch_prefix(b, i) + "offsets must not decrease");
    n_pos[i] = dkb_stream_positions(offsets[i], n_reads[i]);
  }
  return DKB_OK;
}

// The path every submit form takes.  check() is the form's own argument checks; stage(st) is
// the device step of a host form: it puts the batches on the device (in staging slot st) and
// sets b.d_bases / b.d_mask.  The pending loci are used up whatever the outcome.
template <typename Check, typename StageFn>
int submit(dkb_ctx *ctx, const Batches &b, Check check, StageFn stage) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  if (!ctx->d_tslots) return fail(ctx, DKB_ESTATE, "dkb_table_build must come first");
  dkb_ctx::Loci loci[DKB_MAX_MULTI];
  int n_loci = 0, rc;
  if (ctx->regions && (rc = take_loci(ctx, b.multi, loci, n_loci)) != DKB_OK) return rc;
  if ((rc = check()) != DKB_OK) return rc;
  bool any = false;
  for (int i = 0; i < b.n; i++) {
    if (check_sample(ctx, b.samples[i]) != DKB_OK) return DKB_EINVAL;
    if (b.n_positions[i] > 0xFFFFF000ull) return fail(ctx, DKB_EINVAL, "batch too long (max 2^32 - 4096 positions)");
    any |= b.n_positions[i] != 0;
  }
  // (after the form's checks: dkb_batch_submit_reads knows its positions once its offsets are checked)
  if (ctx->regions && (rc = check_loci_positions(ctx, b, loci, n_loci)) != DKB_OK) return rc;
  if (!any) return DKB_OK;
  CU(cudaSetDevice(ctx->device));
  dkb_ctx::Stage *st = nullptr;
  dkb_ctx::LociStage *ls = nullptr;
  if ((rc = stage(st)) != DKB_OK) return rc;
  if (ctx->regions && (rc = stage_loci(ctx, b.n, loci, ls)) != DKB_OK) return rc;
  if ((rc = launch_scan(ctx, b, ls)) != DKB_OK) return rc;
  return release(ctx, {ls, st});
}

// The device step of the device forms: none.
int on_device(dkb_ctx::Stage *&) { return DKB_OK; }

// One batch's loci, as dkb_batch_set_loci takes them, checked and kept in *out.
int check_loci(dkb_ctx *ctx, const uint64_t *offsets, const uint64_t *lo, const uint64_t *hi, size_t n_reads,
               dkb_ctx::Loci *out) {
  if ((uint64_t)n_reads >= 0x100000000ull) return fail(ctx, DKB_EINVAL, "too many reads in one batch (max 2^32 - 1)");
  if (!offsets || (n_reads && (!lo || !hi))) return fail(ctx, DKB_EINVAL, "null loci array");
  for (size_t r = 0; r < n_reads; r++)
    if (offsets[r + 1] < offsets[r]) return fail(ctx, DKB_EINVAL, "offsets must not decrease");
  out->offsets = offsets;
  out->lo = lo;
  out->hi = hi;
  out->n_reads = n_reads;
  out->n_pos = dkb_stream_positions(offsets, n_reads);
  return DKB_OK;
}

// Kernel 3 on snapshot b, on the scan stream, once its sum over ranks is complete.
int finalise_snapshot(dkb_ctx *ctx, const dkb_thresholds *thr, int b) {
  CU(cudaStreamWaitEvent(ctx->s_scan, ctx->ev_red[b], 0));
  int rc = finalise_counts(ctx, thr, ctx->d_red[b], ctx->red_has_cls[b] ? ctx->d_red_cls[b] : nullptr,
                           ctx->red_sexes[b]);
  ctx->red_last = b;
  return rc;
}

}  // namespace

extern "C" {

int dkb_abi_version(void) { return DKB_ABI_VERSION; }

const char *dkb_strerror(int code) {
  switch (code) {
    case DKB_OK: return "ok";
    case DKB_EINVAL: return "invalid argument";
    case DKB_ECUDA: return "CUDA error";
    case DKB_ENOMEM: return "out of memory";
    case DKB_ESTATE: return "call out of order";
    case DKB_ENODEV: return "no usable CUDA device (no CPU fallback exists)";
    case DKB_ENCCL: return "NCCL error";
    default: return "unknown error";
  }
}

const char *dkb_last_error(const dkb_ctx *ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }

int dkb_ctx_create(int device, int k, dkb_ctx **out) { return dkb_ctx_create_family(device, k, 1, out); }

int dkb_ctx_create_family(int device, int k, int n_children, dkb_ctx **out) {
  dkb_ctx *ctx = nullptr;
  if (!out) return fail(nullptr, DKB_EINVAL, "out is null");
  *out = nullptr;
  if (k < DKB_MIN_K || k > DKB_MAX_K) return fail(nullptr, DKB_EINVAL, "k out of range [8, 31]");
  if (n_children < 1 || n_children > DKB_MAX_CHILDREN)
    return fail(nullptr, DKB_EINVAL, "n_children out of range [1, " + std::to_string(DKB_MAX_CHILDREN) + "]");
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
    cudaGetLastError();
    return fail(nullptr, DKB_ENODEV, "no CUDA device; this library has no CPU fallback");
  }
  if (device < 0 || device >= n_dev) return fail(nullptr, DKB_EINVAL, "device index out of range");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess)
    return fail(nullptr, DKB_ECUDA, "cudaGetDeviceProperties failed");
  if (prop.major != 10)
    return fail(nullptr, DKB_ENODEV,
                std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
                    "; kernels are built for sm_100a only");
  ctx = new (std::nothrow) dkb_ctx();
  if (!ctx) return fail(nullptr, DKB_ENOMEM, "host allocation failed");
  ctx->device = device;
  ctx->k = k;
  ctx->n_children = n_children;
  ctx->n_samples = 2 + n_children;
  ctx->n_sms = prop.multiProcessorCount;
  int rc = [&]() -> int {
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&ctx->s_scan, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&ctx->s_copy, cudaStreamNonBlocking));
    for (auto &st : ctx->stage.slot) {
      CU(cudaEventCreateWithFlags(&st.copied, cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&st.freed, cudaEventDisableTiming));
    }
    for (auto &st : ctx->lstage.slot) {
      CU(cudaEventCreateWithFlags(&st.copied, cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&st.freed, cudaEventDisableTiming));
    }
    CU(cudaMalloc(&ctx->d_prof, 4 * sizeof(unsigned long long)));
    CU(cudaMemset(ctx->d_prof, 0, 4 * sizeof(unsigned long long)));
    return DKB_OK;
  }();
  if (rc != DKB_OK) {
    g_err = ctx->err;
    dkb_ctx_destroy(ctx);
    return rc;
  }
  *out = ctx;
  return DKB_OK;
}

int dkb_ctx_destroy(dkb_ctx *ctx) {
  if (!ctx) return DKB_OK;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  free_table(ctx);
  dfree(ctx->d_prof);
  for (auto &st : ctx->stage.slot) st.free();
  for (auto &st : ctx->lstage.slot) st.free();
  for (auto *v : {&ctx->ev_pool, &ctx->ev_pending})
    for (auto &pr : *v) {
      cudaEventDestroy(pr.first);
      cudaEventDestroy(pr.second);
    }
  if (ctx->comm && nccl()->h) nccl()->CommDestroy(ctx->comm);
  for (int i = 0; i < 2; i++) {
    dfree(ctx->d_red[i]);
    if (ctx->ev_snap[i]) cudaEventDestroy(ctx->ev_snap[i]);
    if (ctx->ev_red[i]) cudaEventDestroy(ctx->ev_red[i]);
  }
  if (ctx->s_side) cudaStreamDestroy(ctx->s_side);
  if (ctx->s_scan) cudaStreamDestroy(ctx->s_scan);
  if (ctx->s_copy) cudaStreamDestroy(ctx->s_copy);
  delete ctx;
  return DKB_OK;
}

int dkb_ctx_get_children(const dkb_ctx *ctx, int *n_children_out) {
  if (!ctx || !n_children_out) return fail(nullptr, DKB_EINVAL, "null argument");
  *n_children_out = ctx->n_children;
  return DKB_OK;
}

int dkb_ctx_set_tuning(dkb_ctx *ctx, const dkb_tuning *tuning) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  ctx->user_tuning = tuning ? *tuning : dkb_tuning{0, 0, 0, 0};
  return DKB_OK;
}

int dkb_ctx_get_tuning(const dkb_ctx *ctx, dkb_tuning *out) {
  if (!ctx || !out) return fail(nullptr, DKB_EINVAL, "null argument");
  out->seed_len = ctx->s;
  out->stride = ctx->D;
  out->bloom_hashes = ctx->NH;
  out->filter_mode = ctx->gf ? 2 : 1;
  return DKB_OK;
}

int dkb_table_build(dkb_ctx *ctx, const uint64_t *keys, const uint32_t *variant_ids,
                    const uint8_t *allele_ids, const uint16_t *win_index,
                    const uint16_t *win_count, size_t n, uint32_t n_variants) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  if (n && (!keys || !variant_ids || !allele_ids)) return fail(ctx, DKB_EINVAL, "null entry array");
  if (n >= 0x40000000ull) return fail(ctx, DKB_EINVAL, "too many entries (max 2^30 - 1)");
  if ((win_index == nullptr) != (win_count == nullptr))
    return fail(ctx, DKB_EINVAL, "win_index and win_count must be given together");
  const uint64_t km = kmer_mask(ctx->k);
  for (size_t i = 0; i < n; i++) {
    if (keys[i] > km) return fail(ctx, DKB_EINVAL, "key wider than 2k bits");
    if (variant_ids[i] >= n_variants) return fail(ctx, DKB_EINVAL, "variant id out of range");
    if (allele_ids[i] >= DKB_N_ALLELES) return fail(ctx, DKB_EINVAL, "allele id must be 0 or 1");
    if (win_index && ((win_index[i] & 0x7FFFu) >= win_count[i]))
      return fail(ctx, DKB_EINVAL, "win_index >= win_count");
  }
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->s_scan));
  CU(cudaStreamSynchronize(ctx->s_copy));
  free_table(ctx);
  int rc = resolve_tuning(ctx, n, win_index != nullptr);
  if (rc != DKB_OK) return rc;

  ctx->n_entries = n;
  ctx->n_variants = n_variants;
  const size_t n1 = n ? n : 1, nv1 = n_variants ? n_variants : 1, ns = ctx->n_samples;
  ctx->table_slots = pow2_at_least(8 * (uint64_t)n + 2);  // <= 0.25 entries per 2-slot bucket
  uint16_t *d_wi = nullptr, *d_wc = nullptr;
  uint32_t *d_slot_of = nullptr;
  uint32_t *d_set = nullptr, *d_cov = nullptr, *d_dir = nullptr;
  unsigned int *d_nseeds = nullptr;
  unsigned long long *d_stats = nullptr;
  cudaStream_t st = ctx->s_scan;
  auto cleanup = [&]() {
    dfree(d_wi); dfree(d_wc); dfree(d_slot_of); dfree(d_set); dfree(d_cov); dfree(d_dir); dfree(d_nseeds);
    dfree(d_stats);
  };
  rc = [&]() -> int {
    CU(cudaMalloc(&ctx->d_keys, n1 * 8));
    CU(cudaMalloc(&ctx->d_variant, n1 * 4));
    CU(cudaMalloc(&ctx->d_allele, n1));
    CU(cudaMalloc(&ctx->d_dead, n1));
    CU(cudaMalloc(&d_slot_of, n1 * 4));
    CU(cudaMalloc(&ctx->d_tslots, (size_t)ctx->table_slots * 16));
    CU(cudaMalloc(&ctx->d_counts, n1 * ns * 4));
    // hits, distinct, n_kmers: one block of nv1 * (4 * ns + 2) words, one memset per finalise
    CU(cudaMalloc(&ctx->d_hits, nv1 * (4 * ns + 2) * 4));
    ctx->d_distinct = ctx->d_hits + nv1 * 2 * ns;
    ctx->d_nkmers = ctx->d_hits + nv1 * 4 * ns;
    CU(cudaMalloc(&ctx->d_calls, nv1 * ctx->n_children));
    CU(cudaMalloc(&d_nseeds, 4));
    CU(cudaMemsetAsync(ctx->d_tslots, 0xFF, (size_t)ctx->table_slots * 16, st));
    CU(cudaMemsetAsync(ctx->d_counts, 0, n1 * ns * 4, st));
    CU(cudaMemsetAsync(ctx->d_dead, 0, n1, st));
    CU(cudaMemsetAsync(d_nseeds, 0, 4, st));
    if (n) {
      CU(cudaMemcpyAsync(ctx->d_keys, keys, n * 8, cudaMemcpyHostToDevice, st));
      CU(cudaMemcpyAsync(ctx->d_variant, variant_ids, n * 4, cudaMemcpyHostToDevice, st));
      CU(cudaMemcpyAsync(ctx->d_allele, allele_ids, n, cudaMemcpyHostToDevice, st));
      if (win_index) {
        CU(cudaMalloc(&d_wi, n * 2));
        CU(cudaMalloc(&d_wc, n * 2));
        CU(cudaMemcpyAsync(d_wi, win_index, n * 2, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(d_wc, win_count, n * 2, cudaMemcpyHostToDevice, st));
      }
    }
    // sizing pass: count the distinct seeds in a plain open-addressing set
    const uint32_t set_slots = pow2_at_least(4 * (uint64_t)n * ctx->D + 2);
    CU(cudaMalloc(&d_set, (size_t)set_slots * 4));
    CU(cudaMemsetAsync(d_set, 0xFF, (size_t)set_slots * 4, st));
    BuildParams B;
    B.keys = ctx->d_keys; B.variant = ctx->d_variant; B.allele = ctx->d_allele;
    B.win_index = d_wi; B.win_count = d_wc; B.n = (uint32_t)n;
    B.kt = key_table(ctx); B.slot_of = d_slot_of; B.dead = ctx->d_dead;
    B.k = ctx->k; B.s = ctx->s; B.D = ctx->D;
    // (whether the L2 mode runs behind a pre-filter does not matter here: both are mode > 0)
    ctx->canon = canon_for_mode(ctx->gf ? 1 : 0);
    B.canon = ctx->canon;
    const uint32_t seed_mult = SEED_MULT << (32 - 2 * ctx->s);
    const int TB = 256;
    const uint32_t g1 = (uint32_t)((n + TB - 1) / TB), g2 = (uint32_t)((2 * n + TB - 1) / TB);
    if (n) {
      k_insert_entries<<<g1, TB, 0, st>>>(B);
      k_mark_repeats<<<g1, TB, 0, st>>>(B);
      k_apply_dead<<<g1, TB, 0, st>>>(B);
      k_assign_seeds<<<g2, TB, 0, st>>>(B, ASSIGN_COUNT, d_set, set_slots - 1, d_nseeds, SeedTable{},
                                        nullptr, nullptr, 0, nullptr, 0, seed_mult, ctx->NH, nullptr);
      CU(cudaGetLastError());
    }
    unsigned int n_seeds = 0;
    CU(cudaMemcpyAsync(&n_seeds, d_nseeds, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    ctx->n_seeds = n_seeds;
    dfree(d_set);  // done with: the direct-record scratch below takes its place
    d_set = nullptr;
    // Seed table: 64-byte slots (seed + a 32-byte record per read orientation), a quarter full, any
    // size.  Only occupied slots are ever touched by true hits, so the hot set is 32 B per seed
    // and orientation; an absent seed (a filter false positive) lands on a slot marked
    // ST_MOVED_BIT - a second load - about one time in 8.
    const double per_seed = 4.0;  // (2.0: 3 % slower on configs[1] - displaced seeds cost a dependent load per step)
    const double want_slots = per_seed * n_seeds + 64;
    if (want_slots >= 4294967295.0) return fail(ctx, DKB_EINVAL, "too many seeds for the seed table");
    ctx->seed_slots = (uint32_t)want_slots;
    CU(cudaMalloc(&ctx->d_sslots, (size_t)ctx->seed_slots * 64));
    if (!ctx->gf) {  // probe array: 8 words per seed (dkb_device.cuh)
      const double want_probe = 8.0 * n_seeds + 64;
      if (want_probe >= 4294967295.0) return fail(ctx, DKB_EINVAL, "too many seeds for the probe array");
      ctx->probe_slots = (uint32_t)want_probe;
      CU(cudaMalloc(&ctx->d_probe, (size_t)ctx->probe_slots * 4));
      CU(cudaMemsetAsync(ctx->d_probe, 0x40, (size_t)ctx->probe_slots * 4, st));  // ST_EMPTY
    }
    CU(cudaMalloc(&d_cov, (size_t)ctx->seed_slots * 24));
    CU(cudaMemsetAsync(d_cov, 0, (size_t)ctx->seed_slots * 24, st));
    const size_t dir_bytes = (size_t)ctx->seed_slots * 2 * DIR_WORDS * 4;  // per record half
    CU(cudaMalloc(&d_dir, dir_bytes));
    CU(cudaMemsetAsync(d_dir, 0, dir_bytes, st));
    ctx->bloom_words = ctx->gf ? l2_filter_words((double)n_seeds) / 4 * 4 : (uint32_t)BLOOM_WORDS;
    CU(cudaMalloc(&ctx->d_bloom, (size_t)ctx->bloom_words * 4));
    CU(cudaMemsetAsync(ctx->d_bloom, 0, (size_t)ctx->bloom_words * 4, st));
    ctx->pre_words = ctx->gf ? pre_filter_words(ctx->want_pre) : 0;
    // Gated lookups (macro path of the L2 modes): worth their instructions when most lookups
    // end in an L2 gather - always without a pre-filter, behind one when it passes more than
    // about half (measured, profiles/README.md: 10 000 candidates, 40 % passed: 7.15 -> 6.45
    // Tbases/s; 14 000, 51 %: 5.78 -> 5.83; 20 000, 64 %: 4.52 -> 5.02; no pre-filter: 3.91 -> 6.23).
    ctx->gate = false;
    if (ctx->gf && ctx->D >= 8) {
      const double pass = ctx->pre_words ? 1.0 - exp(-(double)n_seeds / (32.0 * ctx->pre_words)) : 1.0;
      ctx->gate = pass > 0.55;
      if (const char *e = getenv("DKB_GATE")) ctx->gate = atoi(e) != 0;
    }
    if (ctx->pre_words) {
      CU(cudaMalloc(&ctx->d_pre, (size_t)ctx->pre_words * 4));
      CU(cudaMemsetAsync(ctx->d_pre, 0, (size_t)ctx->pre_words * 4, st));
    }
    const SeedTable T = seed_table(ctx);
    k_init_slots<<<(uint32_t)((4 * (size_t)ctx->seed_slots + TB - 1) / TB), TB, 0, st>>>(T);
    // build statistics, counted on the device (the filter can be 16 MB): filter bits set, live
    // entries, occupied record halves, direct ones
    CU(cudaMalloc(&d_stats, 32));
    CU(cudaMemsetAsync(d_stats, 0, 32, st));
    if (n) {
      k_assign_seeds<<<g2, TB, 0, st>>>(B, ASSIGN_INSERT, nullptr, 0, nullptr, T, nullptr,
                                        ctx->d_bloom, ctx->bloom_words, ctx->d_pre, ctx->pre_words,
                                        seed_mult, ctx->NH, nullptr);
      k_assign_seeds<<<g2, TB, 0, st>>>(B, ASSIGN_RECORD, nullptr, 0, nullptr, T, d_cov,
                                        ctx->d_bloom, ctx->bloom_words, ctx->d_pre, ctx->pre_words,
                                        seed_mult, ctx->NH, nullptr);
      const uint32_t gh = (uint32_t)((2 * (size_t)ctx->seed_slots + TB - 1) / TB);
      k_finish_records<<<gh, TB, 0, st>>>(T, d_cov);
      k_assign_seeds<<<g2, TB, 0, st>>>(B, ASSIGN_DIRECT, nullptr, 0, nullptr, T, d_cov,
                                        ctx->d_bloom, ctx->bloom_words, ctx->d_pre, ctx->pre_words,
                                        seed_mult, ctx->NH, d_dir);
      k_finish_direct<<<gh, TB, 0, st>>>(T, d_cov, d_dir, ctx->k, ctx->s, d_stats + 2);
    }
    k_build_stats<<<296, 256, 0, st>>>(ctx->d_bloom, ctx->bloom_words, ctx->d_dead, (uint32_t)n, d_stats);
    CU(cudaGetLastError());
    unsigned long long h_stats[4] = {0, 0, 0, 0};
    CU(cudaMemcpyAsync(h_stats, d_stats, 32, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    ctx->bloom_bits_set = h_stats[0];
    ctx->n_live = (size_t)h_stats[1];
    ctx->occupied_halves = h_stats[2];
    ctx->direct_halves = h_stats[3];
    return DKB_OK;
  }();
  cleanup();
  if (rc != DKB_OK) free_table(ctx);
  return rc;
}

int dkb_batch_submit_device(dkb_ctx *ctx, const uint32_t *d_bases2, const uint32_t *d_mask1,
                            uint64_t n_positions, int sample) {
  const Batches b{false, 1, &n_positions, &sample, &d_bases2, &d_mask1};
  return submit(ctx, b, [&]() -> int { return check_streams(ctx, b, &d_bases2, &d_mask1, true); }, on_device);
}

int dkb_batch_submit_device_multi(dkb_ctx *ctx, int n_batches, const uint32_t *const *d_bases2,
                                  const uint32_t *const *d_mask1, const uint64_t *n_positions,
                                  const int *samples) {
  const Batches b{true, n_batches, n_positions, samples, d_bases2, d_mask1};
  return submit(ctx, b, [&]() -> int { return check_streams(ctx, b, d_bases2, d_mask1, true); }, on_device);
}

int dkb_batch_submit_multi(dkb_ctx *ctx, int n_batches, const uint32_t *const *bases2,
                           const uint32_t *const *mask1, const uint64_t *n_positions, const int *samples) {
  const uint32_t *d_bases[DKB_MAX_MULTI], *d_mask[DKB_MAX_MULTI];
  const Batches b{true, n_batches, n_positions, samples, d_bases, d_mask};
  return submit(ctx, b, [&]() -> int { return check_streams(ctx, b, bases2, mask1, false); },
                [&](dkb_ctx::Stage *&st) { return stage_batches(ctx, b, bases2, mask1, d_bases, d_mask, st); });
}

int dkb_batch_submit(dkb_ctx *ctx, const uint32_t *bases2, const uint32_t *mask1,
                     uint64_t n_positions, int sample) {
  const uint32_t *d_bases, *d_mask;
  const Batches b{false, 1, &n_positions, &sample, &d_bases, &d_mask};
  return submit(ctx, b, [&]() -> int { return check_streams(ctx, b, &bases2, &mask1, false); },
                [&](dkb_ctx::Stage *&st) { return stage_batches(ctx, b, &bases2, &mask1, &d_bases, &d_mask, st); });
}

int dkb_batch_submit_sparse(dkb_ctx *ctx, const uint32_t *bases2, const uint32_t *zoff,
                            const uint8_t *zbytes, size_t zbytes_used, uint64_t n_positions, int sample) {
  const uint32_t *d_bases, *d_mask;
  const Batches b{false, 1, &n_positions, &sample, &d_bases, &d_mask};
  return submit(ctx, b, [&]() -> int { return check_sparse(ctx, b, &bases2, &zoff, &zbytes, &zbytes_used); },
                [&](dkb_ctx::Stage *&st) {
                  return stage_sparse(ctx, b, &bases2, &zoff, &zbytes, &zbytes_used, &d_bases, &d_mask, st);
                });
}

int dkb_batch_submit_sparse_multi(dkb_ctx *ctx, int n_batches, const uint32_t *const *bases2,
                                  const uint32_t *const *zoff, const uint8_t *const *zbytes,
                                  const size_t *zbytes_used, const uint64_t *n_positions, const int *samples) {
  const uint32_t *d_bases[DKB_MAX_MULTI], *d_mask[DKB_MAX_MULTI];
  const Batches b{true, n_batches, n_positions, samples, d_bases, d_mask};
  return submit(ctx, b, [&]() -> int { return check_sparse(ctx, b, bases2, zoff, zbytes, zbytes_used); },
                [&](dkb_ctx::Stage *&st) {
                  return stage_sparse(ctx, b, bases2, zoff, zbytes, zbytes_used, d_bases, d_mask, st);
                });
}

int dkb_batch_submit_reads(dkb_ctx *ctx, const uint8_t *seq, int seq_format, const uint8_t *qual,
                           const uint64_t *offsets, size_t n_reads, int min_baseq, int sample) {
  uint64_t n_pos = 0;  // known once the offsets are checked
  const uint32_t *d_bases, *d_mask;
  const Batches b{false, 1, &n_pos, &sample, &d_bases, &d_mask};
  return submit(ctx, b, [&]() -> int { return check_reads(ctx, b, &seq, seq_format, &offsets, &n_reads, &n_pos); },
                [&](dkb_ctx::Stage *&st) {
                  return stage_reads(ctx, b, &seq, seq_format, &qual, &offsets, &n_reads, min_baseq, &d_bases,
                                     &d_mask, st);
                });
}

int dkb_batch_submit_reads_multi(dkb_ctx *ctx, int n_batches, const uint8_t *const *seq, int seq_format,
                                 const uint8_t *const *qual, const uint64_t *const *offsets,
                                 const size_t *n_reads, int min_baseq, const int *samples) {
  uint64_t n_pos[DKB_MAX_MULTI] = {};  // known once the offsets are checked
  const uint32_t *d_bases[DKB_MAX_MULTI], *d_mask[DKB_MAX_MULTI];
  const Batches b{true, n_batches, n_pos, samples, d_bases, d_mask};
  return submit(ctx, b, [&]() -> int { return check_reads(ctx, b, seq, seq_format, offsets, n_reads, n_pos); },
                [&](dkb_ctx::Stage *&st) {
                  return stage_reads(ctx, b, seq, seq_format, qual, offsets, n_reads, min_baseq, d_bases, d_mask, st);
                });
}

int dkb_table_set_regions(dkb_ctx *ctx, const uint64_t *lo, const uint64_t *hi, uint32_t n_variants) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  if (!ctx->d_tslots) return fail(ctx, DKB_ESTATE, "dkb_table_build must come first");
  drop_loci(ctx);
  if (!lo && !hi) {
    if (n_variants) return fail(ctx, DKB_EINVAL, "lo == hi == NULL (whole-stream counting) takes n_variants 0");
    ctx->regions = false;
    return DKB_OK;
  }
  if (!lo || !hi) return fail(ctx, DKB_EINVAL, "lo and hi must be given together");
  if (n_variants != ctx->n_variants)
    return fail(ctx, DKB_EINVAL, "n_variants differs from the table's (" + std::to_string(ctx->n_variants) + ")");
  CU(cudaSetDevice(ctx->device));
  std::vector<ulonglong2> win(n_variants ? n_variants : 1);
  for (uint32_t v = 0; v < n_variants; v++) win[v] = make_ulonglong2(lo[v], hi[v]);
  const size_t n1 = ctx->n_entries ? ctx->n_entries : 1;
  if (!ctx->d_entry_win) CU(cudaMalloc(&ctx->d_entry_win, n1 * sizeof(ulonglong2)));
  ulonglong2 *d_win = nullptr;
  CU(cudaMalloc(&d_win, win.size() * sizeof(ulonglong2)));
  // on the scan stream: scans queued before this call still read the previous windows
  int rc = [&]() -> int {
    CU(cudaMemcpyAsync(d_win, win.data(), win.size() * sizeof(ulonglong2), cudaMemcpyHostToDevice, ctx->s_scan));
    const int TB = 256;
    if (ctx->n_entries)
      k_entry_windows<<<(uint32_t)((ctx->n_entries + TB - 1) / TB), TB, 0, ctx->s_scan>>>(
          ctx->d_variant, d_win, (uint32_t)ctx->n_entries, ctx->d_entry_win);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->s_scan));
    return DKB_OK;
  }();
  dfree(d_win);
  if (rc != DKB_OK) return rc;
  ctx->regions = true;
  return DKB_OK;
}

int dkb_table_set_locus_classes(dkb_ctx *ctx, const uint8_t *cls, uint32_t n_variants) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  if (!ctx->d_tslots) return fail(ctx, DKB_ESTATE, "dkb_table_build must come first");
  if (!cls) {
    if (n_variants) return fail(ctx, DKB_EINVAL, "cls == NULL (all autosomal) takes n_variants 0");
    ctx->cls_on = false;
    return DKB_OK;
  }
  if (n_variants != ctx->n_variants)
    return fail(ctx, DKB_EINVAL, "n_variants differs from the table's (" + std::to_string(ctx->n_variants) + ")");
  for (uint32_t v = 0; v < n_variants; v++)
    if (cls[v] > DKB_LOCUS_MATERNAL)
      return fail(ctx, DKB_EINVAL, "locus class of variant " + std::to_string(v) + " is above 3");
  CU(cudaSetDevice(ctx->device));
  if (!ctx->d_cls) CU(cudaMalloc(&ctx->d_cls, n_variants ? n_variants : 1));
  // on the scan stream: a kernel 3 queued before this call still reads the previous classes
  if (n_variants) CU(cudaMemcpyAsync(ctx->d_cls, cls, n_variants, cudaMemcpyHostToDevice, ctx->s_scan));
  CU(cudaStreamSynchronize(ctx->s_scan));
  ctx->cls_on = true;
  return DKB_OK;
}

int dkb_ctx_set_child_sexes(dkb_ctx *ctx, const uint8_t *sex, int n_children) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  if (!sex && n_children == 0) n_children = ctx->n_children;
  if (n_children != ctx->n_children)
    return fail(ctx, DKB_EINVAL, "n_children differs from the context's (" + std::to_string(ctx->n_children) + ")");
  ChildSexes s = 0;
  for (int c = 0; sex && c < n_children; c++) {
    if (sex[c] > DKB_SEX_FEMALE) return fail(ctx, DKB_EINVAL, "sex of child " + std::to_string(c) + " is above 2");
    s |= (ChildSexes)sex[c] << (2 * c);
  }
  ctx->sexes = s;
  return DKB_OK;
}

int dkb_batch_set_loci(dkb_ctx *ctx, const uint64_t *offsets, const uint64_t *lo, const uint64_t *hi,
                       size_t n_reads) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  drop_loci(ctx);
  if (!ctx->regions) return fail(ctx, DKB_ESTATE, "dkb_batch_set_loci needs region mode (dkb_table_set_regions)");
  int rc = check_loci(ctx, offsets, lo, hi, n_reads, &ctx->loci[0]);
  if (rc != DKB_OK) return rc;
  ctx->loci_n = 1;
  ctx->loci_multi = false;
  ctx->loci_set = true;
  return DKB_OK;
}

int dkb_batch_set_loci_multi(dkb_ctx *ctx, int n_batches, const uint64_t *const *offsets,
                             const uint64_t *const *lo, const uint64_t *const *hi, const size_t *n_reads) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  drop_loci(ctx);
  if (!ctx->regions) return fail(ctx, DKB_ESTATE, "dkb_batch_set_loci_multi needs region mode (dkb_table_set_regions)");
  if (n_batches < 0 || n_batches > DKB_MAX_MULTI) return fail(ctx, DKB_EINVAL, "n_batches out of range");
  if (n_batches && (!offsets || !lo || !hi || !n_reads)) return fail(ctx, DKB_EINVAL, "null argument");
  uint64_t total = 0;  // reads are numbered across the launch's batches in 32 bits
  for (int i = 0; i < n_batches; i++) {
    int rc = check_loci(ctx, offsets[i], lo[i], hi[i], n_reads[i], &ctx->loci[i]);
    if (rc != DKB_OK) return rc;
    total += n_reads[i];
  }
  if (total >= 0x100000000ull) return fail(ctx, DKB_EINVAL, "too many reads in one launch (max 2^32 - 1)");
  ctx->loci_n = n_batches;
  ctx->loci_multi = true;
  ctx->loci_set = true;
  return DKB_OK;
}

int dkb_sync(dkb_ctx *ctx) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->s_copy));
  CU(cudaStreamSynchronize(ctx->s_scan));
  return DKB_OK;
}

int dkb_counts_reset(dkb_ctx *ctx) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  if (!ctx->d_counts) return fail(ctx, DKB_ESTATE, "dkb_table_build must come first");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemsetAsync(ctx->d_counts, 0, (ctx->n_entries ? ctx->n_entries : 1) * ctx->n_samples * 4, ctx->s_scan));
  if (ctx->prof) CU(cudaMemsetAsync(ctx->d_prof, 0, 4 * sizeof(unsigned long long), ctx->s_scan));
  ctx->finalised = false;
  return DKB_OK;
}

int dkb_entry_counts_fetch(dkb_ctx *ctx, uint32_t *out) {
  if (!ctx || !out) return fail(ctx, DKB_EINVAL, "null argument");
  if (!ctx->d_counts) return fail(ctx, DKB_ESTATE, "dkb_table_build must come first");
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->s_copy));
  CU(cudaMemcpyAsync(out, ctx->d_counts, ctx->n_entries * ctx->n_samples * 4, cudaMemcpyDeviceToHost, ctx->s_scan));
  CU(cudaStreamSynchronize(ctx->s_scan));
  return DKB_OK;
}

int dkb_entry_counts_device(dkb_ctx *ctx, void **d_ptr, size_t *n_u32) {
  if (!ctx || !d_ptr || !n_u32) return fail(ctx, DKB_EINVAL, "null argument");
  if (!ctx->d_counts) return fail(ctx, DKB_ESTATE, "dkb_table_build must come first");
  *d_ptr = ctx->d_counts;
  *n_u32 = ctx->n_entries * ctx->n_samples;
  return DKB_OK;
}

int dkb_finalise(dkb_ctx *ctx, const dkb_thresholds *thr) {
  if (!ctx || !thr) return fail(ctx, DKB_EINVAL, "null argument");
  if (!ctx->d_counts) return fail(ctx, DKB_ESTATE, "dkb_table_build must come first");
  return dkb_finalise_from(ctx, thr, ctx->d_counts);
}

int dkb_finalise_from(dkb_ctx *ctx, const dkb_thresholds *thr, const uint32_t *d_counts) {
  if (!ctx || !thr || !d_counts) return fail(ctx, DKB_EINVAL, "null argument");
  if (!ctx->d_counts) return fail(ctx, DKB_ESTATE, "dkb_table_build must come first");
  CU(cudaSetDevice(ctx->device));
  return finalise_counts(ctx, thr, d_counts, ctx->cls_on ? ctx->d_cls : nullptr, ctx->sexes);
}

}  // extern "C"

namespace {
// Kernel 3 for NS samples.
template <int NS>
void launch_finalise(dkb_ctx *ctx, const Thresholds &T, const uint32_t *d_counts, const uint8_t *cls,
                     const ChildSexes &sexes) {
  cudaStream_t st = ctx->s_scan;
  const int TB = 256;
  if (ctx->n_entries)
    k_variant_reduce<NS><<<(uint32_t)((ctx->n_entries + TB - 1) / TB), TB, 0, st>>>(
        d_counts, ctx->d_variant, ctx->d_allele, ctx->d_dead, (uint32_t)ctx->n_entries,
        ctx->d_hits, ctx->d_distinct, ctx->d_nkmers);
  const uint32_t n_items = ctx->n_variants * (uint32_t)(NS - 2);  // (variant, child) pairs
  if (n_items)
    k_calls<NS><<<(n_items + TB - 1) / TB, TB, 0, st>>>(ctx->d_hits, ctx->d_distinct, n_items, T, cls, sexes,
                                                        ctx->d_calls);
}

int finalise_counts(dkb_ctx *ctx, const dkb_thresholds *thr, const uint32_t *d_counts, const uint8_t *cls,
                    const ChildSexes &sexes) {
  const size_t nv1 = ctx->n_variants ? ctx->n_variants : 1;
  CU(cudaMemsetAsync(ctx->d_hits, 0, nv1 * (4 * (size_t)ctx->n_samples + 2) * 4, ctx->s_scan));
  Thresholds T{thr->min_child_alt_hits, thr->min_child_alt_distinct, thr->max_parent_alt_hits,
               thr->min_parent_ref_hits};
  static_assert(DKB_MAX_CHILDREN == 6, "one kernel-3 instantiation per family size");
  switch (ctx->n_samples) {
    case 3: launch_finalise<3>(ctx, T, d_counts, cls, sexes); break;
    case 4: launch_finalise<4>(ctx, T, d_counts, cls, sexes); break;
    case 5: launch_finalise<5>(ctx, T, d_counts, cls, sexes); break;
    case 6: launch_finalise<6>(ctx, T, d_counts, cls, sexes); break;
    case 7: launch_finalise<7>(ctx, T, d_counts, cls, sexes); break;
    case 8: launch_finalise<8>(ctx, T, d_counts, cls, sexes); break;
    default: return fail(ctx, DKB_EINVAL, "no kernel 3 for this family size");
  }
  CU(cudaGetLastError());
  ctx->finalised = true;
  return DKB_OK;
}
}  // namespace

extern "C" {

// ---- multi-GPU: one sum over ranks of the per-entry counters ---------------------------
int dkb_comm_unique_id(void *id_out) {
  dkb_ctx *ctx = nullptr;
  if (!id_out) return fail(nullptr, DKB_EINVAL, "id_out is null");
  if (!nccl()->h) return fail(nullptr, DKB_ENCCL, "cannot load libnccl.so.2: " + nccl()->err);
  NcclId id;
  NC(nccl()->GetUniqueId(&id));
  memcpy(id_out, &id, sizeof(id));
  return DKB_OK;
}

int dkb_comm_init(dkb_ctx *ctx, const void *id, int rank, int world) {
  if (!ctx || !id) return fail(ctx, DKB_EINVAL, "null argument");
  if (world < 1 || rank < 0 || rank >= world) return fail(ctx, DKB_EINVAL, "rank / world out of range");
  if (ctx->comm) return fail(ctx, DKB_ESTATE, "communicator already initialised");
  if (!nccl()->h) return fail(ctx, DKB_ENCCL, "cannot load libnccl.so.2: " + nccl()->err);
  CU(cudaSetDevice(ctx->device));
  NcclId nid;
  memcpy(&nid, id, sizeof(nid));
  void *comm = nullptr;
  NC(nccl()->CommInitRank(&comm, world, nid, rank));
  ctx->comm = comm;
  ctx->rank = rank;
  ctx->world = world;
  return DKB_OK;
}

int dkb_comm_destroy(dkb_ctx *ctx) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  if (!ctx->comm) return DKB_OK;
  CU(cudaSetDevice(ctx->device));
  if (ctx->s_side) CU(cudaStreamSynchronize(ctx->s_side));
  CU(cudaStreamSynchronize(ctx->s_scan));
  NC(nccl()->CommDestroy(ctx->comm));
  ctx->comm = nullptr;
  ctx->rank = 0;
  ctx->world = 1;
  return DKB_OK;
}

int dkb_comm_info(const dkb_ctx *ctx_c, int *rank, int *world, int *nccl_version) {
  dkb_ctx *ctx = const_cast<dkb_ctx *>(ctx_c);
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  if (rank) *rank = ctx->rank;
  if (world) *world = ctx->world;
  if (world && ctx->comm && nccl()->CommCount) NC(nccl()->CommCount(ctx->comm, world));
  if (nccl_version) {
    *nccl_version = 0;
    if (ctx->comm && nccl()->GetVersion) nccl()->GetVersion(nccl_version);
  }
  return DKB_OK;
}

int dkb_counts_allreduce(dkb_ctx *ctx) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  if (!ctx->d_counts) return fail(ctx, DKB_ESTATE, "dkb_table_build must come first");
  if (!ctx->comm || ctx->world == 1) return DKB_OK;
  CU(cudaSetDevice(ctx->device));
  if (ctx->n_entries)
    NC(nccl()->AllReduce(ctx->d_counts, ctx->d_counts, ctx->n_entries * ctx->n_samples, NCCL_UINT32, NCCL_SUM,
                         ctx->comm, ctx->s_scan));
  ctx->finalised = false;
  return DKB_OK;
}

int dkb_reduce_push(dkb_ctx *ctx, const dkb_thresholds *thr) {
  if (!ctx || !thr) return fail(ctx, DKB_EINVAL, "null argument");
  if (!ctx->d_counts) return fail(ctx, DKB_ESTATE, "dkb_table_build must come first");
  CU(cudaSetDevice(ctx->device));
  int rc = reduce_setup(ctx);
  if (rc != DKB_OK) return rc;
  const int b = ctx->red_next;
  ctx->red_next ^= 1;
  const size_t n = ctx->n_entries * ctx->n_samples;
  // snapshot on the scan stream (behind this batch's scans) ...
  if (n) CU(cudaMemcpyAsync(ctx->d_red[b], ctx->d_counts, n * 4, cudaMemcpyDeviceToDevice, ctx->s_scan));
  CU(cudaEventRecord(ctx->ev_snap[b], ctx->s_scan));
  // ... summed over ranks on the side stream while the scan stream moves on
  CU(cudaStreamWaitEvent(ctx->s_side, ctx->ev_snap[b], 0));
  if (ctx->comm && ctx->world > 1 && n)
    NC(nccl()->AllReduce(ctx->d_red[b], ctx->d_red[b], n, NCCL_UINT32, NCCL_SUM, ctx->comm, ctx->s_side));
  CU(cudaEventRecord(ctx->ev_red[b], ctx->s_side));
  // the classes and sexes in force now go with the snapshot (the copy, on the scan stream, comes
  // after the kernel 3 that last read this buffer)
  ctx->red_has_cls[b] = ctx->cls_on;
  ctx->red_sexes[b] = ctx->sexes;
  if (ctx->cls_on) {
    if (!ctx->d_red_cls[b]) CU(cudaMalloc(&ctx->d_red_cls[b], ctx->n_variants ? ctx->n_variants : 1));
    if (ctx->n_variants)
      CU(cudaMemcpyAsync(ctx->d_red_cls[b], ctx->d_cls, ctx->n_variants, cudaMemcpyDeviceToDevice, ctx->s_scan));
  }
  const int prev = ctx->red_pending;
  ctx->red_pending = b;
  if (prev >= 0) return finalise_snapshot(ctx, thr, prev);
  return DKB_OK;
}

int dkb_reduce_flush(dkb_ctx *ctx, const dkb_thresholds *thr) {
  if (!ctx || !thr) return fail(ctx, DKB_EINVAL, "null argument");
  if (ctx->red_pending < 0) return DKB_OK;
  CU(cudaSetDevice(ctx->device));
  const int b = ctx->red_pending;
  ctx->red_pending = -1;
  return finalise_snapshot(ctx, thr, b);
}

int dkb_reduced_counts_fetch(dkb_ctx *ctx, uint32_t *out) {
  if (!ctx || !out) return fail(ctx, DKB_EINVAL, "null argument");
  if (ctx->red_last < 0) return fail(ctx, DKB_ESTATE, "no reduced batch has been finalised yet");
  CU(cudaSetDevice(ctx->device));
  CU(cudaMemcpyAsync(out, ctx->d_red[ctx->red_last], ctx->n_entries * ctx->n_samples * 4, cudaMemcpyDeviceToHost,
                     ctx->s_scan));
  CU(cudaStreamSynchronize(ctx->s_scan));
  return DKB_OK;
}

int dkb_results_fetch(dkb_ctx *ctx, uint32_t *hits, uint32_t *distinct, uint32_t *n_kmers,
                      uint8_t *calls) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  if (!ctx->finalised) return fail(ctx, DKB_ESTATE, "dkb_finalise must come first");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->s_scan;
  const size_t nv = ctx->n_variants, ns = ctx->n_samples;
  if (hits) CU(cudaMemcpyAsync(hits, ctx->d_hits, nv * 2 * ns * 4, cudaMemcpyDeviceToHost, st));
  if (distinct) CU(cudaMemcpyAsync(distinct, ctx->d_distinct, nv * 2 * ns * 4, cudaMemcpyDeviceToHost, st));
  if (n_kmers) CU(cudaMemcpyAsync(n_kmers, ctx->d_nkmers, nv * 2 * 4, cudaMemcpyDeviceToHost, st));
  if (calls) CU(cudaMemcpyAsync(calls, ctx->d_calls, nv * ctx->n_children, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return DKB_OK;
}

int dkb_stats_get(dkb_ctx *ctx, dkb_stats *out) {
  if (!ctx || !out) return fail(ctx, DKB_EINVAL, "null argument");
  memset(out, 0, sizeof(*out));
  CU(cudaSetDevice(ctx->device));
  out->n_entries = ctx->n_entries;
  out->n_live_entries = ctx->n_live;
  out->table_slots = ctx->table_slots;
  out->n_seeds = ctx->n_seeds;
  out->seed_slots = ctx->seed_slots;
  out->bloom_words = ctx->bloom_words;
  out->bloom_bits_set = ctx->bloom_bits_set;
  out->scan_launches = ctx->scan_launches;
  out->positions_scanned = ctx->positions_scanned;
  CU(cudaStreamSynchronize(ctx->s_scan));
  unsigned long long prof[4];
  CU(cudaMemcpy(prof, ctx->d_prof, sizeof(prof), cudaMemcpyDeviceToHost));
  out->bloom_hits = prof[0];
  out->seed_hits = prof[1];
  out->windows_probed = prof[2];
  out->window_hits = prof[3];
  collect_timing(ctx);
  out->scan_launches_timed = ctx->scan_launches_timed;
  out->scan_ms_total = ctx->scan_ms_total;
  out->last_scan_ms = ctx->last_scan_ms;
  out->prefilter_words = ctx->gf ? ctx->pre_words : 0;
  out->gated_lookups = ctx->gate ? 1u : 0u;
  out->occupied_halves = ctx->occupied_halves;
  out->direct_halves = ctx->direct_halves;
  return DKB_OK;
}

int dkb_profile_counters(dkb_ctx *ctx, int enable) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  if (enable && !ctx->prof) {  // counters start from zero when profiling is switched on
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemsetAsync(ctx->d_prof, 0, 4 * sizeof(unsigned long long), ctx->s_scan));
  }
  ctx->prof = enable != 0;
  return DKB_OK;
}

int dkb_thread_bind_near_gpu(dkb_ctx *ctx, int *numa_node_out) {
  if (!ctx) return fail(nullptr, DKB_EINVAL, "ctx is null");
  const int node = gpu_numa_node(ctx->device);
  if (numa_node_out) *numa_node_out = node;
  cpu_set_t set;
  if (node >= 0 && node_cpus(node, &set)) sched_setaffinity(0, sizeof(set), &set);  // best effort
  return DKB_OK;
}

int dkb_host_alloc(dkb_ctx *ctx, size_t bytes, void **out) {
  if (!ctx || !out) return fail(ctx, DKB_EINVAL, "null argument");
  *out = nullptr;
  CU(cudaSetDevice(ctx->device));
  // allocate (and thereby pin: the pages are populated at once) while this thread runs on,
  // and prefers memory of, the NUMA node the GPU hangs off; then put the thread back
  const int node = gpu_numa_node(ctx->device);
  cpu_set_t old, near;
  const bool have_old = sched_getaffinity(0, sizeof(old), &old) == 0;
  const bool moved = node >= 0 && node_cpus(node, &near) && sched_setaffinity(0, sizeof(near), &near) == 0;
  if (node >= 0) prefer_node(node);
  void *p = nullptr;
  const cudaError_t e = cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault);
  if (node >= 0) prefer_node(-1);
  if (moved && have_old) sched_setaffinity(0, sizeof(old), &old);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(ctx, DKB_ENOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
  }
  *out = p;
  return DKB_OK;
}

int dkb_host_free(dkb_ctx *ctx, void *p) {
  if (!p) return DKB_OK;
  if (ctx) cudaSetDevice(ctx->device);
  if (cudaFreeHost(p) != cudaSuccess) {
    cudaGetLastError();
    return fail(ctx, DKB_ECUDA, "cudaFreeHost failed");
  }
  return DKB_OK;
}

int dkb_scan_stream(dkb_ctx *ctx, void **stream_out) {
  if (!ctx || !stream_out) return fail(ctx, DKB_EINVAL, "null argument");
  *stream_out = (void *)ctx->s_scan;
  return DKB_OK;
}

}  // extern "C"

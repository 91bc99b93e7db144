// dkb.hpp — header-only C++17 convenience layer over the C ABI in dkb.h: RAII context,
// std::vector in/out, exceptions instead of error codes.  Nothing here computes; every
// call forwards to libdkb.so.  (The reference is a Rust crate — INTEGRATION.md shows its
// binding; this is the same surface for C++ hosts and for this repo's own C++ tests.)
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "dkb.h"

namespace dkbxx {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string &what) : std::runtime_error(what), code(c) {}
};

inline void check(int rc, const dkb_ctx *ctx = nullptr) {
  if (rc != DKB_OK)
    throw Error(rc, std::string(dkb_strerror(rc)) + ": " + dkb_last_error(ctx));
}

// Spanning k-mer entries of a candidate list (counter.rs: per-allele k-mer sets).
struct Entries {
  std::vector<uint64_t> keys;
  std::vector<uint32_t> variant;
  std::vector<uint8_t> allele;
  std::vector<uint16_t> win_index, win_count;
  uint32_t n_variants = 0;
};

struct Candidate {
  std::string left, ref, alt, right;  // flanks hold at least k-1 reference bases each
};

inline Entries variant_kmers(const std::vector<Candidate> &c, int k, bool drop_shared = true) {
  std::vector<const char *> l, r, a, rt;
  for (const auto &v : c) {
    l.push_back(v.left.c_str());
    r.push_back(v.ref.c_str());
    a.push_back(v.alt.c_str());
    rt.push_back(v.right.c_str());
  }
  size_t n = 0;
  check(dkb_variant_kmers(l.data(), r.data(), a.data(), rt.data(), c.size(), k, drop_shared, nullptr,
                          nullptr, nullptr, nullptr, nullptr, &n));
  Entries e;
  e.keys.resize(n);
  e.variant.resize(n);
  e.allele.resize(n);
  e.win_index.resize(n);
  e.win_count.resize(n);
  e.n_variants = (uint32_t)c.size();
  check(dkb_variant_kmers(l.data(), r.data(), a.data(), rt.data(), c.size(), k, drop_shared,
                          e.keys.data(), e.variant.data(), e.allele.data(), e.win_index.data(),
                          e.win_count.data(), &n));
  return e;
}

// Packed read stream (kmer.rs: what the per-read k-mer iteration consumes).
struct Stream {
  std::vector<uint32_t> bases2, mask1;
  uint64_t n_positions = 0;
};

// four_bit: seq holds BAM 4-bit codes (high nibble first, every read on a byte boundary)
inline Stream pack_reads(const std::vector<uint8_t> &seq, const std::vector<uint8_t> &qual,
                         const std::vector<uint64_t> &offsets, int min_baseq, bool four_bit = false) {
  const size_t n_reads = offsets.empty() ? 0 : offsets.size() - 1;
  Stream s;
  s.n_positions = dkb_stream_positions(offsets.data(), n_reads);
  s.bases2.resize(dkb_stream_bases_words(s.n_positions) + 1);
  s.mask1.resize(dkb_stream_mask_words(s.n_positions) + 1);
  check(dkb_pack_reads_fmt(seq.data(), four_bit ? 1 : 0, qual.empty() ? nullptr : qual.data(), offsets.data(),
                           n_reads, min_baseq, s.bases2.data(), s.mask1.data(), &s.n_positions));
  return s;
}

struct Results {
  std::vector<uint32_t> hits, distinct;  // [n_variants][2 alleles][n_samples]
  std::vector<uint32_t> n_kmers;         // [n_variants][2]
  std::vector<uint8_t> calls;            // [n_variants][n_children], DKB_CALL_* bits
};

// One GPU context.  Throws Error{DKB_ENODEV} when no sm_100 device exists: there is no
// CPU fallback.  n_children > 1: a family (dkb_ctx_create_family) - mother 1, father 2, child
// c at DKB_CHILD_SAMPLE(c), n_samples() = 2 + n_children.
class Counter {
 public:
  Counter(int k, int device = 0, int n_children = 1) : n_children_(n_children) {
    check(dkb_ctx_create_family(device, k, n_children, &ctx_));
  }
  ~Counter() { dkb_ctx_destroy(ctx_); }
  Counter(const Counter &) = delete;
  Counter &operator=(const Counter &) = delete;

  void set_tuning(const dkb_tuning &t) { check(dkb_ctx_set_tuning(ctx_, &t), ctx_); }
  void build_table(const Entries &e) {
    check(dkb_table_build(ctx_, e.keys.data(), e.variant.data(), e.allele.data(),
                          e.win_index.empty() ? nullptr : e.win_index.data(),
                          e.win_count.empty() ? nullptr : e.win_count.data(), e.keys.size(),
                          e.n_variants),
          ctx_);
    n_entries_ = e.keys.size();
    n_variants_ = e.n_variants;
  }
  // the stream must outlive the next sync()
  void submit(const Stream &s, int sample) {
    check(dkb_batch_submit(ctx_, s.bases2.data(), s.mask1.data(), s.n_positions, sample), ctx_);
  }
  // decoded reads packed on the GPU (ASCII bases, or BAM 4-bit codes when four_bit)
  void submit_reads(const std::vector<uint8_t> &seq, const std::vector<uint8_t> &qual,
                    const std::vector<uint64_t> &offsets, int min_baseq, int sample,
                    bool four_bit = false) {
    check(dkb_batch_submit_reads(ctx_, seq.data(), four_bit ? 1 : 0, qual.empty() ? nullptr : qual.data(),
                                 offsets.data(), offsets.empty() ? 0 : offsets.size() - 1, min_baseq,
                                 sample),
          ctx_);
  }
  // the stream with its flags as a zero list (dkb_mask_to_zero_list): less PCIe traffic;
  // the vectors must outlive the next sync()
  struct SparseStream {
    std::vector<uint32_t> bases2, zoff;
    std::vector<uint8_t> zbytes;
    uint64_t n_positions = 0;
  };
  static SparseStream to_sparse(const Stream &s) {
    SparseStream z;
    z.bases2 = s.bases2;
    z.n_positions = s.n_positions;
    z.zoff.resize(dkb_zero_list_blocks(s.n_positions) + 1);
    size_t used = 0;
    check(dkb_mask_to_zero_list(s.mask1.data(), s.n_positions, z.zoff.data(), nullptr, 0, &used));
    z.zbytes.resize(used + 1);
    check(dkb_mask_to_zero_list(s.mask1.data(), s.n_positions, z.zoff.data(), z.zbytes.data(), used, &used));
    z.zbytes.resize(used);
    return z;
  }
  void submit(const SparseStream &z, int sample) {
    check(dkb_batch_submit_sparse(ctx_, z.bases2.data(), z.zoff.data(), z.zbytes.data(), z.zbytes.size(),
                                  z.n_positions, sample),
          ctx_);
  }
  // multi-GPU: one context per GPU and rank; id from dkb_comm_unique_id on rank 0
  void comm_init(const void *id, int rank, int world) { check(dkb_comm_init(ctx_, id, rank, world), ctx_); }
  void counts_allreduce() { check(dkb_counts_allreduce(ctx_), ctx_); }
  void reduce_push(const dkb_thresholds &t) { check(dkb_reduce_push(ctx_, &t), ctx_); }
  void reduce_flush(const dkb_thresholds &t) { check(dkb_reduce_flush(ctx_, &t), ctx_); }
  // Region mode (dkb.h): a read counts toward variant v only if its alignment interval
  // overlaps [lo[v], hi[v]); every later submit needs set_loci() first.
  void set_regions(const std::vector<uint64_t> &lo, const std::vector<uint64_t> &hi) {
    if (lo.size() != hi.size()) throw Error(DKB_EINVAL, "set_regions: lo and hi differ in length");
    check(dkb_table_set_regions(ctx_, lo.data(), hi.data(), (uint32_t)lo.size()), ctx_);
  }
  void clear_regions() { check(dkb_table_set_regions(ctx_, nullptr, nullptr, 0), ctx_); }
  // Inheritance (dkb.h): the locus class of every variant (DKB_LOCUS_*) and the sex of every
  // child (DKB_SEX_*) decide which parents' clauses each call applies.
  void set_locus_classes(const std::vector<uint8_t> &cls) {
    check(dkb_table_set_locus_classes(ctx_, cls.data(), (uint32_t)cls.size()), ctx_);
  }
  void clear_locus_classes() { check(dkb_table_set_locus_classes(ctx_, nullptr, 0), ctx_); }
  void set_child_sexes(const std::vector<uint8_t> &sex) {
    check(dkb_ctx_set_child_sexes(ctx_, sex.data(), (int)sex.size()), ctx_);
  }
  // The loci of the next submit: the batch's offsets and its reads' [lo, hi).  The vectors
  // must stay alive and unchanged until sync().
  void set_loci(const std::vector<uint64_t> &offsets, const std::vector<uint64_t> &lo,
                const std::vector<uint64_t> &hi) {
    if (offsets.empty() || lo.size() + 1 != offsets.size() || hi.size() != lo.size())
      throw Error(DKB_EINVAL, "set_loci: lo and hi need one entry per read");
    check(dkb_batch_set_loci(ctx_, offsets.data(), lo.data(), hi.data(), lo.size()), ctx_);
  }
  // Loci of the next multi-batch submit, one set per batch (each as in set_loci); same lifetime rule.
  struct LociRef {
    const std::vector<uint64_t> *offsets, *lo, *hi;
  };
  void set_loci_multi(const std::vector<LociRef> &loci) {
    std::vector<const uint64_t *> o, l, h;
    std::vector<size_t> n;
    for (const LociRef &x : loci) {
      if (x.offsets->empty() || x.lo->size() + 1 != x.offsets->size() || x.hi->size() != x.lo->size())
        throw Error(DKB_EINVAL, "set_loci_multi: lo and hi need one entry per read");
      o.push_back(x.offsets->data());
      l.push_back(x.lo->data());
      h.push_back(x.hi->data());
      n.push_back(x.lo->size());
    }
    check(dkb_batch_set_loci_multi(ctx_, (int)loci.size(), o.data(), l.data(), h.data(), n.data()), ctx_);
  }
  // Up to DKB_MAX_MULTI streams, (stream, sample), in ONE scan launch (a trio step); the streams
  // must outlive the next sync()
  void submit_multi(const std::vector<std::pair<const Stream *, int>> &batches) {
    std::vector<const uint32_t *> b, m;
    std::vector<uint64_t> n;
    std::vector<int> smp;
    for (const auto &x : batches) {
      b.push_back(x.first->bases2.data());
      m.push_back(x.first->mask1.data());
      n.push_back(x.first->n_positions);
      smp.push_back(x.second);
    }
    check(dkb_batch_submit_multi(ctx_, (int)batches.size(), b.data(), m.data(), n.data(), smp.data()), ctx_);
  }
  // Up to DKB_MAX_MULTI zero-list streams, (stream, sample), in one expand and ONE scan launch;
  // the streams must outlive the next sync()
  void submit_sparse_multi(const std::vector<std::pair<const SparseStream *, int>> &batches) {
    std::vector<const uint32_t *> b, z;
    std::vector<const uint8_t *> zb;
    std::vector<size_t> used;
    std::vector<uint64_t> n;
    std::vector<int> smp;
    for (const auto &x : batches) {
      b.push_back(x.first->bases2.data());
      z.push_back(x.first->zoff.data());
      zb.push_back(x.first->zbytes.data());
      used.push_back(x.first->zbytes.size());
      n.push_back(x.first->n_positions);
      smp.push_back(x.second);
    }
    check(dkb_batch_submit_sparse_multi(ctx_, (int)batches.size(), b.data(), z.data(), zb.data(), used.data(),
                                        n.data(), smp.data()),
          ctx_);
  }
  // One batch of decoded reads for submit_reads_multi (as in submit_reads; qual may be empty)
  struct ReadsRef {
    const std::vector<uint8_t> *seq, *qual;
    const std::vector<uint64_t> *offsets;
    int sample;
  };
  // Up to DKB_MAX_MULTI batches of decoded reads in one pack and ONE scan launch; the vectors
  // must outlive the next sync()
  void submit_reads_multi(const std::vector<ReadsRef> &batches, int min_baseq, bool four_bit = false) {
    std::vector<const uint8_t *> s, q;
    std::vector<const uint64_t *> o;
    std::vector<size_t> nr;
    std::vector<int> smp;
    for (const ReadsRef &x : batches) {
      s.push_back(x.seq->data());
      q.push_back(x.qual->empty() ? nullptr : x.qual->data());
      o.push_back(x.offsets->data());
      nr.push_back(x.offsets->empty() ? 0 : x.offsets->size() - 1);
      smp.push_back(x.sample);
    }
    check(dkb_batch_submit_reads_multi(ctx_, (int)batches.size(), s.data(), four_bit ? 1 : 0, q.data(), o.data(),
                                       nr.data(), min_baseq, smp.data()),
          ctx_);
  }
  void sync() { check(dkb_sync(ctx_), ctx_); }
  void reset_counts() { check(dkb_counts_reset(ctx_), ctx_); }
  int n_children() const { return n_children_; }
  size_t n_samples() const { return 2 + (size_t)n_children_; }
  std::vector<uint32_t> entry_counts() {  // [n_samples][n_entries]
    std::vector<uint32_t> out(n_samples() * n_entries_ + 1);
    check(dkb_entry_counts_fetch(ctx_, out.data()), ctx_);
    out.resize(n_samples() * n_entries_);
    return out;
  }
  // d_counts: optional caller-owned DEVICE copy of the counters (dkb_finalise_from)
  Results finalise(const dkb_thresholds &t, const uint32_t *d_counts = nullptr) {
    check(d_counts ? dkb_finalise_from(ctx_, &t, d_counts) : dkb_finalise(ctx_, &t), ctx_);
    Results r;
    const size_t nh = 2 * n_samples() * n_variants_, nc = (size_t)n_children_ * n_variants_;
    r.hits.resize(nh + 1);
    r.distinct.resize(nh + 1);
    r.n_kmers.resize(2 * (size_t)n_variants_ + 1);
    r.calls.resize(nc + 1);
    check(dkb_results_fetch(ctx_, r.hits.data(), r.distinct.data(), r.n_kmers.data(), r.calls.data()),
          ctx_);
    r.hits.resize(nh);
    r.distinct.resize(nh);
    r.n_kmers.resize(2 * (size_t)n_variants_);
    r.calls.resize(nc);
    return r;
  }
  dkb_ctx *raw() { return ctx_; }

 private:
  dkb_ctx *ctx_ = nullptr;
  int n_children_ = 1;
  size_t n_entries_ = 0;
  uint32_t n_variants_ = 0;
};

}  // namespace dkbxx

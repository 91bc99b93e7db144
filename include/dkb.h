/*
 * dkb.h — C ABI of the B200-native de novo k-mer hot path (libdkb.so).
 *
 * Drop-in boundary for jlanej/denovo_kmer's one data-parallel path:
 *   src/kmer.rs     k-mer extraction + canonical hashing from child/parent reads
 *   src/counter.rs  membership counting against each candidate allele's
 *                   spanning k-mer set, per sample (child / mother / father)
 *   (caller)        de novo support thresholds
 * Those files are NOT in the /root/reference mount (SURVEY.md §0: only
 * .github/workflows/ci.yml:1-50 and .gitignore:1 are); the semantics this
 * ABI implements are therefore the ones written down in DESIGN.md §2
 * ("spec"), which follows BASELINE.json `north_star`.  Parity is UNPINNED
 * against the real reference until its source is mounted.
 *
 * Conventions
 *   - every function returns DKB_OK (0) or a DKB_E* code; nothing throws or
 *     aborts across the ABI; dkb_last_error(ctx) has the detail string.
 *   - caller owns every host buffer; the library owns all device memory.
 *   - one context per GPU, one submitting thread per context.
 *   - there is NO CPU fallback: without a CUDA device dkb_ctx_create fails
 *     with DKB_ENODEV.
 *   - base codes: A=0 C=1 G=2 T=3.  A k-mer value ("key") packs the first
 *     base in the most significant of its 2k bits; canonical = min(fwd, rc).
 *
 * Packed read batch ("stream") — what src/kmer.rs would iterate, as bits:
 *   bases2 : uint32 words, 16 bases each, base p in bits 2*(p%16) of word p/16
 *   mask1  : uint32 words, 32 flags each, flag p in bit  p%32     of word p/32
 *            flag = 1 iff base p is A/C/G/T and its base quality >= min_baseq
 *   every read is followed by ONE separator position with flag 0, so the
 *   rolling window resets at read ends exactly like an N does.
 *   n_positions = sum(read lengths) + n_reads.  A k-mer at position w counts
 *   iff flags w..w+k-1 are all 1.
 */
#ifndef DKB_H
#define DKB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DKB_ABI_VERSION 1
#define DKB_MIN_K 8
#define DKB_MAX_K 31
#define DKB_N_SAMPLES 3 /* 0 child, 1 mother, 2 father */
/* Family contexts (dkb_ctx_create_family): one mother, one father and n_children children counted
 * against one table, NS = 2 + n_children samples.  Mother stays sample 1 and father sample 2, so
 * a one-child family IS a trio.  Every array laid out with DKB_N_SAMPLES below holds NS samples
 * in a family context. */
#define DKB_MAX_CHILDREN 6 /* a family has at most 2 + 6 = 8 samples */
/* sample index of child c (0 <= c < n_children): 0 for c == 0, else 2 + c */
#define DKB_CHILD_SAMPLE(c) ((c) == 0 ? 0 : (c) + 2)
#define DKB_N_ALLELES 2 /* 0 ref, 1 alt (multi-allelic sites are split by the host) */

enum {
  DKB_OK = 0,
  DKB_EINVAL = 1, /* bad argument */
  DKB_ECUDA = 2,  /* CUDA runtime error (see dkb_last_error) */
  DKB_ENOMEM = 3, /* host or device allocation failed */
  DKB_ESTATE = 4, /* call out of order (e.g. submit before table_build) */
  DKB_ENODEV = 5, /* no usable sm_100 device; there is no CPU fallback */
  DKB_ENCCL = 6   /* NCCL error, or libnccl.so.2 cannot be loaded (multi-GPU calls only) */
};

typedef struct dkb_ctx dkb_ctx;

/* De novo support rule (integer only), applied once per child of a family: the clauses
 * name that child's alt hits and distinct k-mers, and both parents' hits.  A variant is
 * called (bit 0 of the call byte) iff
 *   child  alt hits     >= min_child_alt_hits      and
 *   child  alt distinct >= min_child_alt_distinct  and
 *   mother alt hits     <= max_parent_alt_hits     and
 *   father alt hits     <= max_parent_alt_hits     and
 *   mother ref hits     >= min_parent_ref_hits     and
 *   father ref hits     >= min_parent_ref_hits.
 * Failing clauses set bits 1..4 (see DKB_CALL_*).  With locus classes and child sexes set
 * (dkb_table_set_locus_classes, dkb_ctx_set_child_sexes) only the clauses of the parents who can
 * transmit the locus to that child apply; see "inheritance" below. */
typedef struct dkb_thresholds {
  uint32_t min_child_alt_hits;
  uint32_t min_child_alt_distinct;
  uint32_t max_parent_alt_hits;
  uint32_t min_parent_ref_hits;
} dkb_thresholds;

#define DKB_CALL_DENOVO 0x01u         /* all clauses hold */
#define DKB_CALL_CHILD_LOW 0x02u      /* child alt support below minimum */
#define DKB_CALL_MOTHER_ALT 0x04u     /* mother carries alt k-mers */
#define DKB_CALL_FATHER_ALT 0x08u     /* father carries alt k-mers */
#define DKB_CALL_PARENT_UNCOVERED 0x10u /* a parent lacks ref k-mer coverage */
#define DKB_CALL_NO_COPY 0x20u        /* the child's sex has no copy of the locus (a daughter at Y) */

/* Locus class of a variant (dkb_table_set_locus_classes) */
#define DKB_LOCUS_AUTOSOMAL 0 /* autosomes, and PAR1 / PAR2 of X and Y */
#define DKB_LOCUS_X 1         /* X outside the PARs */
#define DKB_LOCUS_Y 2         /* Y outside the PARs */
#define DKB_LOCUS_MATERNAL 3  /* mitochondrial */
/* Sex of a child (dkb_ctx_set_child_sexes) */
#define DKB_SEX_UNKNOWN 0
#define DKB_SEX_MALE 1
#define DKB_SEX_FEMALE 2

/* Scan tuning, normally left to the library (dkb_ctx_set_tuning(ctx, NULL)). */
typedef struct dkb_tuning {
  int seed_len;     /* s: 8..15 and <= k - stride + 1; 0 = auto */
  int stride;       /* D: probe every D-th stream position (1, 2, 4, 8 or 16); 0 = auto */
  int bloom_hashes; /* 1..4 bits per seed in the seed filter; 0 = auto */
  int filter_mode;  /* 1 = filter in shared memory (small candidate sets), 2 = filter in L2
                       (strides 2..16, 1..2 hashes; the library decides whether a 145 KB
                       (37 120-word) shared-memory pre-filter goes in front of it, env
                       DKB_PREFILTER_WORDS overrides); 0 = auto */
} dkb_tuning;

/* ---- library ---------------------------------------------------------- */
int dkb_abi_version(void);
const char *dkb_strerror(int code);
const char *dkb_last_error(const dkb_ctx *ctx);

/* ---- context ---------------------------------------------------------- */
/* A trio: dkb_ctx_create_family(device, k, 1, out). */
int dkb_ctx_create(int device, int k, dkb_ctx **out);
/* A family of n_children children (1..DKB_MAX_CHILDREN; DKB_EINVAL otherwise, checked before
 * the device) and both parents.  Submits take sample in [0, NS): DKB_CHILD_SAMPLE(c) for child
 * c, 1 for the mother, 2 for the father. */
int dkb_ctx_create_family(int device, int k, int n_children, dkb_ctx **out);
int dkb_ctx_get_children(const dkb_ctx *ctx, int *n_children_out);
int dkb_ctx_destroy(dkb_ctx *ctx);
int dkb_ctx_set_tuning(dkb_ctx *ctx, const dkb_tuning *tuning);
int dkb_ctx_get_tuning(const dkb_ctx *ctx, dkb_tuning *out);

/* ---- kmer.rs host-side primitives (pure functions, no device) ----------- */
/* seq[0..k) -> forward key; DKB_EINVAL if a base is not A/C/G/T (either case) */
int dkb_kmer_encode(const char *seq, int k, uint64_t *fwd_out);
uint64_t dkb_kmer_revcomp(uint64_t fwd, int k);
uint64_t dkb_kmer_canonical(uint64_t fwd, int k);

/* ---- host packer: decoded reads -> packed stream ------------------------ */
/* reads are concatenated in seq/qual; read r occupies [offsets[r], offsets[r+1]).
 * qual may be NULL (all qualities pass).  Sizes: */
uint64_t dkb_stream_positions(const uint64_t *offsets, size_t n_reads);
size_t dkb_stream_bases_words(uint64_t n_positions);
size_t dkb_stream_mask_words(uint64_t n_positions);
int dkb_pack_reads(const uint8_t *seq, const uint8_t *qual, const uint64_t *offsets,
                   size_t n_reads, int min_baseq, uint32_t *bases2, uint32_t *mask1,
                   uint64_t *n_positions_out);
/* The same from either form the BAM layer holds (seq_format as in dkb_batch_submit_reads): 0 =
 * ASCII bases, read r at seq[offsets[r]..offsets[r+1]); 1 = BAM 4-bit codes (=ACMGRSVTWYHKDBN,
 * high nibble first: record.seq().encoded of rust-htslib, no decode pass), every read starting
 * on a byte boundary with (len + 1) / 2 bytes, reads back to back from seq[0].  qual is one byte
 * per base at qual[offsets[r]..] either way.  Same stream, bit for bit, for the same reads. */
int dkb_pack_reads_fmt(const uint8_t *seq, int seq_format, const uint8_t *qual, const uint64_t *offsets,
                       size_t n_reads, int min_baseq, uint32_t *bases2, uint32_t *mask1,
                       uint64_t *n_positions_out);

/* ---- the flags as a ZERO LIST (a third less PCIe traffic) ----------------------- */
/* mask1 costs 1 bit per position; with ~4 % of the positions unusable (N, low quality, read
 * separators) it is cheaper to send WHERE the zeros are.  Per block of 2048 positions: a byte
 * string, each byte g < 255 = "g usable positions, then one unusable one", 255 = "255 usable
 * positions" (no zero); positions after the last byte's zero are usable.  A block whose string
 * would exceed 256 bytes is stored as its 256 bytes of plain flag bits instead.  zoff[b] =
 * byte offset of block b's string in zbytes, bit 31 set for a plain-bits block; zoff[n_blocks]
 * = total bytes.  Flags at positions >= n_positions are not coded (the scan ignores them).
 * dkb_mask_to_zero_list converts dense flags (zbytes == NULL: only sizes: *zbytes_used and
 * zoff are filled in); zoff holds dkb_zero_list_blocks(n) + 1 entries. */
size_t dkb_zero_list_blocks(uint64_t n_positions);
int dkb_mask_to_zero_list(const uint32_t *mask1, uint64_t n_positions, uint32_t *zoff, uint8_t *zbytes,
                          size_t zbytes_cap, size_t *zbytes_used);

/* ---- host variant k-mer builder (counter.rs "spanning k-mer set") ------- */
/* For variant v with left flank L, right flank R (reference bases either side
 * of REF, at least k-1 each unless the contig ends) and alleles REF/ALT,
 * haplotype(a) = L[-(k-1):] + allele(a) + R[:k-1]; its spanning k-mers are the
 * windows that overlap the allele, or that straddle the junction when the
 * allele is empty.  Windows with a non-ACGT base are skipped.  Keys present
 * in both alleles of one variant are dropped when drop_shared != 0.  Within one
 * (variant, allele) a key is emitted once (first window wins).
 * Pass keys == NULL to size the output; *n_out returns the entry count.
 * win_index/win_count (may be NULL) give each entry's window index within its
 * haplotype's spanning run and that run's length (seed-ladder hints for
 * dkb_table_build). */
int dkb_variant_kmers(const char *const *left, const char *const *ref,
                      const char *const *alt, const char *const *right, size_t n_variants,
                      int k, int drop_shared, uint64_t *keys, uint32_t *variant_ids,
                      uint8_t *allele_ids, uint16_t *win_index, uint16_t *win_count,
                      size_t *n_out);

/* ---- kernel 1: table build ------------------------------------------------ */
/* Entry i = (canonical key, variant id, allele id); counts are reported per
 * entry index.  A (key, variant, allele) triple repeated in the input keeps
 * its first entry live; later repeats stay at 0.  One key may belong to many
 * (variant, allele) owners: every owner is counted.  win_index/win_count may
 * be NULL. */
int dkb_table_build(dkb_ctx *ctx, const uint64_t *keys, const uint32_t *variant_ids,
                    const uint8_t *allele_ids, const uint16_t *win_index,
                    const uint16_t *win_count, size_t n_entries, uint32_t n_variants);

/* ---- kernel 2: streaming extract-and-probe ------------------------------- */
/* Host buffers (pinned for full speed); H2D copy + scan are queued on the
 * context's streams and overlap with the next submit.  The buffers must stay
 * valid until dkb_sync.  sample: 0..2 in a trio, [0, NS) in a family (DKB_EINVAL otherwise),
 * in every submit form below. */
int dkb_batch_submit(dkb_ctx *ctx, const uint32_t *bases2, const uint32_t *mask1,
                     uint64_t n_positions, int sample);
/* Same as dkb_batch_submit with the flags as a zero list (above): bases2 + zoff + zbytes cross
 * PCIe - 0.29 instead of 0.38 bytes per base at 4 % unusable positions - and the library
 * expands the list into mask1 on the device before the scan. */
int dkb_batch_submit_sparse(dkb_ctx *ctx, const uint32_t *bases2, const uint32_t *zoff,
                            const uint8_t *zbytes, size_t zbytes_used, uint64_t n_positions, int sample);
/* Decoded reads as the BAM layer holds them: the packing (what dkb_pack_reads does on the
 * host) runs on the GPU.  seq_format 0: ASCII bases, read r at seq[offsets[r]..offsets[r+1]);
 * 1: BAM 4-bit codes (=ACMGRSVTWYHKDBN, high nibble first), every read starting on a byte
 * boundary with (len + 1) / 2 bytes, reads back to back from seq[0].  qual (may be NULL):
 * one byte per base at qual[offsets[r]..].  Same stream, bit for bit, as dkb_pack_reads. */
int dkb_batch_submit_reads(dkb_ctx *ctx, const uint8_t *seq, int seq_format, const uint8_t *qual,
                           const uint64_t *offsets, size_t n_reads, int min_baseq, int sample);
/* Device-resident buffers: d_bases2 16-byte aligned, d_mask1 4-byte aligned, each
 * dkb_stream_*_words long.  Flags at positions >= n_positions are ignored. */
int dkb_batch_submit_device(dkb_ctx *ctx, const uint32_t *d_bases2, const uint32_t *d_mask1,
                            uint64_t n_positions, int sample);
/* Up to DKB_MAX_MULTI device-resident streams (e.g. the three samples of a trio, or a quad's four) in ONE kernel
 * launch; batch i goes into the counters of samples[i].  Same alignment rules; a batch of 0
 * positions is skipped.  Worth it for short batches, where a launch costs as much as the scan. */
#define DKB_MAX_MULTI 4
/* In region mode (below) it needs the loci of dkb_batch_set_loci_multi first. */
int dkb_batch_submit_device_multi(dkb_ctx *ctx, int n_batches, const uint32_t *const *d_bases2,
                                  const uint32_t *const *d_mask1, const uint64_t *n_positions,
                                  const int *samples);
/* Up to DKB_MAX_MULTI host-resident batches scanned in ONE kernel launch; batch i goes into the
 * counters of samples[i].  Same buffer rules as dkb_batch_submit: valid until dkb_sync.  A batch
 * of 0 positions is skipped; n_batches 0 is a no-op.  The batches are copied into one staging
 * buffer, each with its own copy, and double-buffered like dkb_batch_submit: a trio step is one
 * submit and one scan launch.  In region mode it needs the loci of dkb_batch_set_loci_multi
 * first. */
int dkb_batch_submit_multi(dkb_ctx *ctx, int n_batches, const uint32_t *const *bases2,
                           const uint32_t *const *mask1, const uint64_t *n_positions, const int *samples);
/* dkb_batch_submit_sparse for up to DKB_MAX_MULTI host-resident batches: batch i is bases2[i]
 * with its flags as the zero list zoff[i] / zbytes[i] / zbytes_used[i], n_positions[i] long, into
 * the counters of samples[i].  Every zero list is checked as dkb_batch_submit_sparse checks it;
 * one launch expands them all, then one scan launch counts them.  The call follows the rules of
 * dkb_batch_submit_multi (n_batches in [0, DKB_MAX_MULTI], empty batches skipped, buffers valid
 * until dkb_sync, the loci of dkb_batch_set_loci_multi in region mode).  A refusal that concerns
 * one batch names it ("batch i: ..."). */
int dkb_batch_submit_sparse_multi(dkb_ctx *ctx, int n_batches, const uint32_t *const *bases2,
                                  const uint32_t *const *zoff, const uint8_t *const *zbytes,
                                  const size_t *zbytes_used, const uint64_t *n_positions, const int *samples);
/* dkb_batch_submit_reads for up to DKB_MAX_MULTI batches of decoded reads: batch i is
 * seq[i] / qual[i] / offsets[i] with n_reads[i] reads, into the counters of samples[i], each under
 * the rules of dkb_batch_submit_reads.  One seq_format and one min_baseq apply to every batch.
 * qual may be NULL (no batch has qualities), and so may any qual[i].  One launch packs every
 * batch, then one scan launch counts them.  The call follows the rules of dkb_batch_submit_multi;
 * a batch of 0 reads is skipped.  A refusal that concerns one batch names it ("batch i: ..."). */
int dkb_batch_submit_reads_multi(dkb_ctx *ctx, int n_batches, const uint8_t *const *seq, int seq_format,
                                 const uint8_t *const *qual, const uint64_t *const *offsets,
                                 const size_t *n_reads, int min_baseq, const int *samples);

/* ---- region-scoped counting (opt-in; DESIGN.md §2) ---------------------------- */
/* In region mode an occurrence of entry e's key in read r counts iff the read's alignment
 * interval [rlo, rhi) overlaps the window [lo, hi) of e's variant (both half-open, in one
 * linear coordinate system the caller chooses, e.g. contig offset + 0-based position).  An
 * empty interval (rlo >= rhi: an unmapped read) or an empty window (lo >= hi) overlaps nothing.
 * Counters, finalise and the multi-GPU sum are unchanged.
 * After dkb_table_build: variant v's window is [lo[v], hi[v]), n_variants as built.
 * lo == hi == NULL (n_variants 0) returns to whole-stream counting.  A new
 * dkb_table_build also returns to it.  DKB_ESTATE before dkb_table_build; DKB_EINVAL if
 * n_variants differs from the table's.  Scans queued earlier keep the windows they were
 * submitted with. */
int dkb_table_set_regions(dkb_ctx *ctx, const uint64_t *lo, const uint64_t *hi, uint32_t n_variants);
/* The read loci of the NEXT single-batch submit (dkb_batch_submit, _sparse, _reads, _device).
 * offsets: n_reads + 1 entries as given to the packer (read r's first base is at stream
 * position offsets[r] - offsets[0] + r).  lo/hi: the reads' alignment intervals.  Copied by
 * that submit with the batch; the buffers follow the submit's validity rule (dkb_batch_submit:
 * valid until dkb_sync; for _device too).  In region mode a single-batch submit without loci
 * returns DKB_ESTATE, and one whose loci cover a different number of stream positions
 * (dkb_stream_positions(offsets, n_reads) != n_positions) DKB_EINVAL; every submit uses up the
 * pending loci whatever its outcome.  DKB_ESTATE in whole-stream mode; DKB_EINVAL for descending
 * offsets or n_reads >= 2^32.  Region mode has no profiling counters: with dkb_profile_counters
 * on, a submit returns DKB_ESTATE. */
int dkb_batch_set_loci(dkb_ctx *ctx, const uint64_t *offsets, const uint64_t *lo,
                       const uint64_t *hi, size_t n_reads);
/* Region mode: the read loci of the NEXT multi-batch submit (dkb_batch_submit_multi,
 * _device_multi, _sparse_multi or _reads_multi), one set per batch, with the same meaning and validity rules
 * as dkb_batch_set_loci.  DKB_ESTATE in whole-stream mode; DKB_EINVAL for n_batches outside
 * [0, DKB_MAX_MULTI], descending offsets in any batch, n_reads[i] >= 2^32, or 2^32 or more
 * reads in all.  The submit returns DKB_EINVAL unless its n_batches equals these loci's and
 * dkb_stream_positions(offsets[i], n_reads[i]) == n_positions[i] for every batch.  Loci of the
 * wrong kind are refused with DKB_ESTATE: a single-batch submit with multi-batch loci pending,
 * a multi-batch submit with single-batch loci pending.  Setting either kind replaces whatever
 * was pending, and every submit uses up the pending loci whatever its outcome. */
int dkb_batch_set_loci_multi(dkb_ctx *ctx, int n_batches, const uint64_t *const *offsets,
                             const uint64_t *const *lo, const uint64_t *const *hi, const size_t *n_reads);
int dkb_sync(dkb_ctx *ctx);
int dkb_counts_reset(dkb_ctx *ctx);

/* per-entry counts, layout [DKB_N_SAMPLES][n_entries]; [NS][n_entries] in a family */
int dkb_entry_counts_fetch(dkb_ctx *ctx, uint32_t *out);
/* device pointer of the same array, for the multi-GPU sum (NCCL allreduce); *n_u32 =
 * NS * n_entries */
int dkb_entry_counts_device(dkb_ctx *ctx, void **d_ptr, size_t *n_u32);

/* ---- kernel 3: finalise ---------------------------------------------------- */
/* Per (variant, allele, sample) hits saturate at UINT32_MAX: a sum past 2^32 - 1 reads as
 * UINT32_MAX, never as its wrapped remainder.  The calls therefore equal the de novo rule on the
 * exact sums for every max_parent_alt_hits below UINT32_MAX and every min_child_alt_hits and
 * min_parent_ref_hits. */
int dkb_finalise(dkb_ctx *ctx, const dkb_thresholds *thr);
/* Same, from a caller-owned DEVICE copy of the counters ([DKB_N_SAMPLES][n_entries], or
   [NS][n_entries] in a family: the layout of dkb_entry_counts_device) - e.g. a copy that is being summed over ranks while
   the context's own counters already take the next batch.  Runs on the scan stream: order
   it after the copy is complete (dkb_scan_stream). */
int dkb_finalise_from(dkb_ctx *ctx, const dkb_thresholds *thr, const uint32_t *d_counts);
/* hits / distinct: [n_variants][DKB_N_ALLELES][DKB_N_SAMPLES] ([n_variants][2][NS] in a
 * family); n_kmers: [n_variants][DKB_N_ALLELES]; calls: [n_variants][n_children], child c's
 * byte at calls[v * n_children + c] (a trio: [n_variants]).  Any pointer may be NULL. */
int dkb_results_fetch(dkb_ctx *ctx, uint32_t *hits, uint32_t *distinct, uint32_t *n_kmers,
                      uint8_t *calls);

/* ---- inheritance: which parents can transmit a locus (opt-in; DESIGN.md §2) ----------- */
/* With nothing set every variant is autosomal and every child's sex unknown: the rule above
 * applies both parents' clauses to every call.  Otherwise, for variant v of class cls[v] and
 * child c of sex sex[c], only these parents' clauses apply ("M": DKB_CALL_MOTHER_ALT and the
 * mother's half of DKB_CALL_PARENT_UNCOVERED; "F": the father's):
 *   class \ sex   unknown  male  female
 *   autosomal     M F      M F   M F
 *   X             M F      M     M F
 *   Y             M F      F     none, and DKB_CALL_NO_COPY is set
 *   maternal      M        M     M
 * DKB_CALL_CHILD_LOW is unchanged, and bit 0 (DKB_CALL_DENOVO) is set iff no other bit is, so a
 * DKB_CALL_NO_COPY byte is never a call.  Thresholds and counting are unchanged.
 * dkb_finalise / dkb_finalise_from use the classes and sexes in force when called;
 * dkb_reduce_push records them with its snapshot, and that snapshot's kernel 3 (queued by the
 * next push or the flush) uses what was recorded.  A kernel 3 already queued never sees a later
 * change.  Multi-GPU: every rank computes the calls from the same summed counters, so every
 * rank must set the same classes and sexes; no collective is involved. */
/* After dkb_table_build: cls[v] in 0..3 (DKB_LOCUS_*) for each of the table's n_variants.
 * cls == NULL (n_variants 0) returns to all-autosomal; so does a new dkb_table_build.
 * DKB_ESTATE before dkb_table_build; DKB_EINVAL if n_variants differs from the table's or a
 * class is above 3. */
int dkb_table_set_locus_classes(dkb_ctx *ctx, const uint8_t *cls, uint32_t n_variants);
/* sex[c] in 0..2 (DKB_SEX_*) for each of the context's n_children children; sex == NULL
 * (n_children 0 or the context's) returns every child to unknown.  Any time; kept across table
 * builds.  DKB_EINVAL if n_children differs from the context's or a sex is above 2. */
int dkb_ctx_set_child_sexes(dkb_ctx *ctx, const uint8_t *sex, int n_children);

/* ---- pinned staging next to the GPU ------------------------------------------ */
/* Page-locked host memory for the packed batches, allocated on the NUMA node the GPU's PCIe
 * slot belongs to (the calling thread is moved there for the allocation and moved back).  With
 * eight ranks pushing batches at once, buffers on the wrong socket halve the H2D rate.
 * dkb_thread_bind_near_gpu pins the CALLING thread (the one that packs and submits) to that
 * node's CPUs for good; *numa_node_out (may be NULL) gets the node, -1 if unknown. */
int dkb_host_alloc(dkb_ctx *ctx, size_t bytes, void **out);
int dkb_host_free(dkb_ctx *ctx, void *p);
int dkb_thread_bind_near_gpu(dkb_ctx *ctx, int *numa_node_out);

/* ---- multi-GPU: read batches sharded over ranks, ONE sum of the counters ------ */
/* One process (or thread) per GPU, each with its own context and its own slice of the read
 * batches; the table is built identically on every rank.  The per-entry counters are summed
 * over ranks with a single NCCL allreduce (libnccl.so.2 is loaded on first use; without it
 * these calls return DKB_ENCCL and everything else works).
 *   rank 0: dkb_comm_unique_id(id)  -> send the DKB_COMM_ID_BYTES to every rank (MPI, TCP, a file ...)
 *   all   : dkb_comm_init(ctx, id, rank, world)
 * Simple form: scan, then dkb_counts_allreduce (in place, on the scan stream), dkb_finalise.
 * Overlapped form, for a sequence of independent batches (trios, regions): after a batch's
 * scans dkb_reduce_push snapshots the counters and starts the sum on a side stream; the
 * caller resets the counters and submits the next batch at once; the push of batch i also
 * queues kernel 3 for batch i-1 behind the scans just submitted, by which time that sum has
 * long finished.  dkb_reduce_flush finalises the last batch; dkb_results_fetch then returns
 * its results and dkb_reduced_counts_fetch its summed counters.  With no communicator (one
 * GPU) both forms run without NCCL and equal plain dkb_finalise. */
#define DKB_COMM_ID_BYTES 128
int dkb_comm_unique_id(void *id_out);
int dkb_comm_init(dkb_ctx *ctx, const void *id, int rank, int world);
int dkb_comm_destroy(dkb_ctx *ctx);
/* rank, communicator size as NCCL reports it, NCCL version (0 without a communicator) */
int dkb_comm_info(const dkb_ctx *ctx, int *rank, int *world, int *nccl_version);
int dkb_counts_allreduce(dkb_ctx *ctx);
int dkb_reduce_push(dkb_ctx *ctx, const dkb_thresholds *thr);
int dkb_reduce_flush(dkb_ctx *ctx, const dkb_thresholds *thr);
/* [DKB_N_SAMPLES][n_entries], [NS][n_entries] in a family */
int dkb_reduced_counts_fetch(dkb_ctx *ctx, uint32_t *out);

/* ---- introspection (bench / tests) --------------------------------------- */
typedef struct dkb_stats {
  uint64_t n_entries, n_live_entries, table_slots;
  uint64_t n_seeds, seed_slots, bloom_words, bloom_bits_set;
  uint64_t scan_launches;    /* scan kernels launched since create */
  uint64_t positions_scanned;
  uint64_t bloom_hits, seed_hits, windows_probed, window_hits; /* if profiling counters on */
  uint64_t scan_launches_timed; /* launches folded into scan_ms_total */
  double scan_ms_total;      /* sum of per-launch CUDA-event times of the scan kernel */
  float last_scan_ms;        /* CUDA-event time of the most recent finished scan kernel */
  uint32_t prefilter_words;  /* L2 filter mode: words of the shared-memory pre-filter, 0 = none */
  uint32_t gated_lookups;    /* 1: the scan also reads the flag stream in full and skips the lookups of
                                seeds that hold an unusable base (env DKB_GATE=0/1 overrides) */
  uint64_t occupied_halves;  /* seed-record halves (one per seed and read orientation) with a designation */
  uint64_t direct_halves;    /* of those, the ones whose windows the scan counts straight from the
                                record, without the key table (DESIGN.md §4) */
} dkb_stats;
int dkb_stats_get(dkb_ctx *ctx, dkb_stats *out);
int dkb_profile_counters(dkb_ctx *ctx, int enable);
/* CUDA stream the scan kernels are launched on (cudaStream_t as void*). */
int dkb_scan_stream(dkb_ctx *ctx, void **stream_out);

#ifdef __cplusplus
}
#endif
#endif /* DKB_H */

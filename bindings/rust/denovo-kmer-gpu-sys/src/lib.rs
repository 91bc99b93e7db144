//! Raw bindings to `libdkb.so` - mirror of `include/dkb.h`, ABI version 1.
//! Every function returns `DKB_OK` (0) or an error code; `dkb_last_error(ctx)` has the text.
//! There is no CPU fallback: `dkb_ctx_create` returns `DKB_ENODEV` without an sm_100 device.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct DkbCtx { _private: [u8; 0] }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct DkbThresholds {
    pub min_child_alt_hits: u32, pub min_child_alt_distinct: u32,
    pub max_parent_alt_hits: u32, pub min_parent_ref_hits: u32,
}
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct DkbTuning { pub seed_len: c_int, pub stride: c_int, pub bloom_hashes: c_int, pub filter_mode: c_int }

#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct DkbStats {
    pub n_entries: u64, pub n_live_entries: u64, pub table_slots: u64,
    pub n_seeds: u64, pub seed_slots: u64, pub bloom_words: u64, pub bloom_bits_set: u64,
    pub scan_launches: u64, pub positions_scanned: u64,
    pub bloom_hits: u64, pub seed_hits: u64, pub windows_probed: u64, pub window_hits: u64,
    pub scan_launches_timed: u64,
    pub scan_ms_total: f64, pub last_scan_ms: f32, pub prefilter_words: u32, pub gated_lookups: u32,
    pub occupied_halves: u64, pub direct_halves: u64,
}

pub const DKB_ABI_VERSION: c_int = 1;
pub const DKB_OK: c_int = 0;
pub const DKB_EINVAL: c_int = 1;
pub const DKB_ECUDA: c_int = 2;
pub const DKB_ENOMEM: c_int = 3;
pub const DKB_ESTATE: c_int = 4;
pub const DKB_ENODEV: c_int = 5;
pub const DKB_ENCCL: c_int = 6;
pub const DKB_COMM_ID_BYTES: usize = 128;
pub const DKB_MAX_MULTI: usize = 4;
pub const DKB_N_SAMPLES: usize = 3;
/// A family context holds at most 2 + DKB_MAX_CHILDREN samples.
pub const DKB_MAX_CHILDREN: usize = 6;
/// Sample index of child `c` in a family (DKB_CHILD_SAMPLE): 0 for c == 0, else 2 + c.
pub const fn dkb_child_sample(c: usize) -> usize { if c == 0 { 0 } else { c + 2 } }
pub const DKB_CALL_DENOVO: u8 = 0x01;
pub const DKB_CALL_CHILD_LOW: u8 = 0x02;
pub const DKB_CALL_MOTHER_ALT: u8 = 0x04;
pub const DKB_CALL_FATHER_ALT: u8 = 0x08;
pub const DKB_CALL_PARENT_UNCOVERED: u8 = 0x10;
/// The child's sex has no copy of the locus (a daughter at Y).
pub const DKB_CALL_NO_COPY: u8 = 0x20;
pub const DKB_LOCUS_AUTOSOMAL: u8 = 0;
pub const DKB_LOCUS_X: u8 = 1;
pub const DKB_LOCUS_Y: u8 = 2;
pub const DKB_LOCUS_MATERNAL: u8 = 3;
pub const DKB_SEX_UNKNOWN: u8 = 0;
pub const DKB_SEX_MALE: u8 = 1;
pub const DKB_SEX_FEMALE: u8 = 2;

extern "C" {
    pub fn dkb_abi_version() -> c_int;
    pub fn dkb_strerror(code: c_int) -> *const c_char;
    pub fn dkb_last_error(ctx: *const DkbCtx) -> *const c_char;
    pub fn dkb_ctx_create(device: c_int, k: c_int, out: *mut *mut DkbCtx) -> c_int;
    pub fn dkb_ctx_create_family(device: c_int, k: c_int, n_children: c_int, out: *mut *mut DkbCtx) -> c_int;
    pub fn dkb_ctx_get_children(ctx: *const DkbCtx, n_children_out: *mut c_int) -> c_int;
    pub fn dkb_ctx_destroy(ctx: *mut DkbCtx) -> c_int;
    pub fn dkb_ctx_set_tuning(ctx: *mut DkbCtx, t: *const DkbTuning) -> c_int;
    pub fn dkb_ctx_get_tuning(ctx: *const DkbCtx, out: *mut DkbTuning) -> c_int;
    pub fn dkb_kmer_encode(seq: *const c_char, k: c_int, fwd_out: *mut u64) -> c_int;
    pub fn dkb_kmer_revcomp(fwd: u64, k: c_int) -> u64;
    pub fn dkb_kmer_canonical(fwd: u64, k: c_int) -> u64;
    pub fn dkb_stream_positions(offsets: *const u64, n_reads: usize) -> u64;
    pub fn dkb_stream_bases_words(n_positions: u64) -> usize;
    pub fn dkb_stream_mask_words(n_positions: u64) -> usize;
    pub fn dkb_pack_reads(seq: *const u8, qual: *const u8, offsets: *const u64, n_reads: usize,
                          min_baseq: c_int, bases2: *mut u32, mask1: *mut u32,
                          n_positions_out: *mut u64) -> c_int;
    pub fn dkb_pack_reads_fmt(seq: *const u8, seq_format: c_int, qual: *const u8, offsets: *const u64,
                              n_reads: usize, min_baseq: c_int, bases2: *mut u32, mask1: *mut u32,
                              n_positions_out: *mut u64) -> c_int;
    pub fn dkb_zero_list_blocks(n_positions: u64) -> usize;
    pub fn dkb_mask_to_zero_list(mask1: *const u32, n_positions: u64, zoff: *mut u32, zbytes: *mut u8,
                                 zbytes_cap: usize, zbytes_used: *mut usize) -> c_int;
    pub fn dkb_variant_kmers(left: *const *const c_char, r#ref: *const *const c_char,
                             alt: *const *const c_char, right: *const *const c_char,
                             n_variants: usize, k: c_int, drop_shared: c_int, keys: *mut u64,
                             variant_ids: *mut u32, allele_ids: *mut u8, win_index: *mut u16,
                             win_count: *mut u16, n_out: *mut usize) -> c_int;
    pub fn dkb_table_build(ctx: *mut DkbCtx, keys: *const u64, variant_ids: *const u32,
                           allele_ids: *const u8, win_index: *const u16, win_count: *const u16,
                           n_entries: usize, n_variants: u32) -> c_int;
    pub fn dkb_batch_submit(ctx: *mut DkbCtx, bases2: *const u32, mask1: *const u32,
                            n_positions: u64, sample: c_int) -> c_int;
    pub fn dkb_batch_submit_sparse(ctx: *mut DkbCtx, bases2: *const u32, zoff: *const u32, zbytes: *const u8,
                                   zbytes_used: usize, n_positions: u64, sample: c_int) -> c_int;
    pub fn dkb_batch_submit_reads(ctx: *mut DkbCtx, seq: *const u8, seq_format: c_int, qual: *const u8,
                                  offsets: *const u64, n_reads: usize, min_baseq: c_int, sample: c_int) -> c_int;
    pub fn dkb_batch_submit_device(ctx: *mut DkbCtx, d_bases2: *const u32, d_mask1: *const u32,
                                   n_positions: u64, sample: c_int) -> c_int;
    pub fn dkb_batch_submit_device_multi(ctx: *mut DkbCtx, n_batches: c_int, d_bases2: *const *const u32,
                                         d_mask1: *const *const u32, n_positions: *const u64,
                                         samples: *const c_int) -> c_int;
    pub fn dkb_table_set_regions(ctx: *mut DkbCtx, lo: *const u64, hi: *const u64, n_variants: u32) -> c_int;
    pub fn dkb_batch_set_loci(ctx: *mut DkbCtx, offsets: *const u64, lo: *const u64, hi: *const u64,
                              n_reads: usize) -> c_int;
    pub fn dkb_batch_submit_multi(ctx: *mut DkbCtx, n_batches: c_int, bases2: *const *const u32,
                                  mask1: *const *const u32, n_positions: *const u64, samples: *const c_int) -> c_int;
    pub fn dkb_batch_submit_sparse_multi(ctx: *mut DkbCtx, n_batches: c_int, bases2: *const *const u32,
                                         zoff: *const *const u32, zbytes: *const *const u8,
                                         zbytes_used: *const usize, n_positions: *const u64,
                                         samples: *const c_int) -> c_int;
    pub fn dkb_batch_submit_reads_multi(ctx: *mut DkbCtx, n_batches: c_int, seq: *const *const u8, seq_format: c_int,
                                        qual: *const *const u8, offsets: *const *const u64, n_reads: *const usize,
                                        min_baseq: c_int, samples: *const c_int) -> c_int;
    pub fn dkb_batch_set_loci_multi(ctx: *mut DkbCtx, n_batches: c_int, offsets: *const *const u64,
                                    lo: *const *const u64, hi: *const *const u64, n_reads: *const usize) -> c_int;
    pub fn dkb_sync(ctx: *mut DkbCtx) -> c_int;
    pub fn dkb_counts_reset(ctx: *mut DkbCtx) -> c_int;
    pub fn dkb_entry_counts_fetch(ctx: *mut DkbCtx, out: *mut u32) -> c_int;
    pub fn dkb_entry_counts_device(ctx: *mut DkbCtx, d_ptr: *mut *mut c_void, n_u32: *mut usize) -> c_int;
    pub fn dkb_finalise(ctx: *mut DkbCtx, thr: *const DkbThresholds) -> c_int;
    pub fn dkb_finalise_from(ctx: *mut DkbCtx, thr: *const DkbThresholds, d_counts: *const u32) -> c_int;
    pub fn dkb_results_fetch(ctx: *mut DkbCtx, hits: *mut u32, distinct: *mut u32,
                             n_kmers: *mut u32, calls: *mut u8) -> c_int;
    pub fn dkb_table_set_locus_classes(ctx: *mut DkbCtx, cls: *const u8, n_variants: u32) -> c_int;
    pub fn dkb_ctx_set_child_sexes(ctx: *mut DkbCtx, sex: *const u8, n_children: c_int) -> c_int;
    pub fn dkb_host_alloc(ctx: *mut DkbCtx, bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn dkb_host_free(ctx: *mut DkbCtx, p: *mut c_void) -> c_int;
    pub fn dkb_thread_bind_near_gpu(ctx: *mut DkbCtx, numa_node_out: *mut c_int) -> c_int;
    pub fn dkb_comm_unique_id(id_out: *mut c_void) -> c_int;
    pub fn dkb_comm_init(ctx: *mut DkbCtx, id: *const c_void, rank: c_int, world: c_int) -> c_int;
    pub fn dkb_comm_destroy(ctx: *mut DkbCtx) -> c_int;
    pub fn dkb_comm_info(ctx: *const DkbCtx, rank: *mut c_int, world: *mut c_int,
                         nccl_version: *mut c_int) -> c_int;
    pub fn dkb_counts_allreduce(ctx: *mut DkbCtx) -> c_int;
    pub fn dkb_reduce_push(ctx: *mut DkbCtx, thr: *const DkbThresholds) -> c_int;
    pub fn dkb_reduce_flush(ctx: *mut DkbCtx, thr: *const DkbThresholds) -> c_int;
    pub fn dkb_reduced_counts_fetch(ctx: *mut DkbCtx, out: *mut u32) -> c_int;
    pub fn dkb_stats_get(ctx: *mut DkbCtx, out: *mut DkbStats) -> c_int;
    pub fn dkb_profile_counters(ctx: *mut DkbCtx, enable: c_int) -> c_int;
    pub fn dkb_scan_stream(ctx: *mut DkbCtx, stream_out: *mut *mut c_void) -> c_int;
}

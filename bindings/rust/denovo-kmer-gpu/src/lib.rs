//! Safe wrapper over `denovo-kmer-gpu-sys` (`include/dkb.h`): what the reference's
//! `counter.rs` would hold instead of its CPU k-mer map.
//!
//! * [`Counter`] owns one GPU context (RAII: `Drop` destroys it), one per GPU and per
//!   submitting thread (`!Sync`; it may be moved to another thread).
//! * every call returns `Result<_, DkbError>`; nothing panics across the FFI boundary.
//! * [`BatchPacker`] turns decoded reads (what `kmer.rs` iterates) into the packed 2-bit
//!   stream inside page-locked buffers next to the GPU, two of them so that packing batch
//!   i + 1 overlaps the copy and scan of batch i.
//! * multi-GPU: [`comm_unique_id`], [`Counter::comm_init`], [`Counter::reduce_push`] - the one
//!   NCCL all-reduce of the per-entry counters is made inside `libdkb.so`.
//!
//! NOT COMPILED in this repository's build container (no Rust toolchain there); kept in step
//! with the header by `tests/test_host.py` (every `dkb_*` call used here must exist in the
//! `-sys` crate with the same arity).
use denovo_kmer_gpu_sys as sys;
use std::ffi::{CStr, CString};
use std::marker::PhantomData;
use std::os::raw::{c_char, c_int, c_void};
use std::ptr;

pub use sys::{DkbStats as Stats, DkbThresholds as Thresholds, DkbTuning as Tuning};

pub const CHILD: i32 = 0;
pub const MOTHER: i32 = 1;
pub const FATHER: i32 = 2;
pub const CALL_DENOVO: u8 = 0x01;
pub const CALL_NO_COPY: u8 = 0x20;

/// Locus class of a candidate (`include/dkb.h` DKB_LOCUS_*), from the VCF's CHROM and POS and
/// the assembly's PAR coordinates.
#[derive(Debug, Clone, Copy, PartialEq, Eq)]
#[repr(u8)]
pub enum LocusClass {
    /// Autosomes, and PAR1 / PAR2 of X and Y.
    Autosomal = 0,
    /// X outside the PARs.
    X = 1,
    /// Y outside the PARs.
    Y = 2,
    /// Mitochondrial.
    Maternal = 3,
}

/// Sex of a child (`include/dkb.h` DKB_SEX_*), from the PED file's sex column.
#[derive(Debug, Clone, Copy, PartialEq, Eq)]
#[repr(u8)]
pub enum Sex {
    Unknown = 0,
    Male = 1,
    Female = 2,
}
pub use sys::{dkb_child_sample as child_sample, DKB_MAX_CHILDREN as MAX_CHILDREN};

/// Error code of the C ABI plus the library's detail string.
#[derive(Debug, Clone)]
pub struct DkbError {
    pub code: i32,
    pub detail: String,
}

impl std::fmt::Display for DkbError {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result {
        let what = unsafe { CStr::from_ptr(sys::dkb_strerror(self.code)) }.to_string_lossy();
        write!(f, "dkb error {} ({}): {}", self.code, what, self.detail)
    }
}
impl std::error::Error for DkbError {}

pub type Result<T> = std::result::Result<T, DkbError>;

fn check(code: c_int, ctx: *const sys::DkbCtx) -> Result<()> {
    if code == sys::DKB_OK {
        return Ok(());
    }
    let p = unsafe { sys::dkb_last_error(ctx) };
    let detail = if p.is_null() { String::new() } else { unsafe { CStr::from_ptr(p) }.to_string_lossy().into_owned() };
    Err(DkbError { code, detail })
}

/// Spanning k-mer entries of the candidate alleles (`counter.rs`'s k-mer set), as the host
/// builder `dkb_variant_kmers` emits them.
#[derive(Default, Clone)]
pub struct Entries {
    pub keys: Vec<u64>,
    pub variant: Vec<u32>,
    pub allele: Vec<u8>,
    pub win_index: Vec<u16>,
    pub win_count: Vec<u16>,
    pub n_variants: u32,
}

/// One candidate: reference flanks either side of REF (k-1 bases each unless the contig ends).
pub struct Candidate<'a> {
    pub left: &'a str,
    pub r#ref: &'a str,
    pub alt: &'a str,
    pub right: &'a str,
}

/// `dkb_variant_kmers`: spanning k-mers of every candidate's REF and ALT haplotype.
pub fn variant_kmers(cands: &[Candidate<'_>], k: i32, drop_shared: bool) -> Result<Entries> {
    fn own<'a>(it: impl Iterator<Item = &'a str>) -> Vec<CString> {
        it.map(|s| CString::new(s).expect("no NUL in sequence")).collect()
    }
    let (l, r, a, t) = (own(cands.iter().map(|c| c.left)), own(cands.iter().map(|c| c.r#ref)),
                        own(cands.iter().map(|c| c.alt)), own(cands.iter().map(|c| c.right)));
    let ptrs = |v: &Vec<CString>| -> Vec<*const c_char> { v.iter().map(|s| s.as_ptr()).collect() };
    let (lp, rp, ap, tp) = (ptrs(&l), ptrs(&r), ptrs(&a), ptrs(&t));
    let mut n: usize = 0;
    check(unsafe {
        sys::dkb_variant_kmers(lp.as_ptr(), rp.as_ptr(), ap.as_ptr(), tp.as_ptr(), cands.len(), k,
                               drop_shared as c_int, ptr::null_mut(), ptr::null_mut(), ptr::null_mut(),
                               ptr::null_mut(), ptr::null_mut(), &mut n)
    }, ptr::null())?;
    let mut e = Entries { keys: vec![0; n], variant: vec![0; n], allele: vec![0; n], win_index: vec![0; n],
                          win_count: vec![0; n], n_variants: cands.len() as u32 };
    check(unsafe {
        sys::dkb_variant_kmers(lp.as_ptr(), rp.as_ptr(), ap.as_ptr(), tp.as_ptr(), cands.len(), k,
                               drop_shared as c_int, e.keys.as_mut_ptr(), e.variant.as_mut_ptr(),
                               e.allele.as_mut_ptr(), e.win_index.as_mut_ptr(), e.win_count.as_mut_ptr(), &mut n)
    }, ptr::null())?;
    Ok(e)
}

/// Per-variant results of kernel 3 (`n_samples` = 3 for a trio, 2 + `n_children` for a family).
pub struct Results {
    /// `[n_variants][allele 0..2][sample 0..n_samples]`
    pub hits: Vec<u32>,
    pub distinct: Vec<u32>,
    /// `[n_variants][allele 0..2]`
    pub n_kmers: Vec<u32>,
    /// `DKB_CALL_*` bits, `[n_variants][child 0..n_children]` (one per variant for a trio)
    pub calls: Vec<u8>,
}

/// One GPU context: table, streams, counters.  One per GPU, used from one thread at a time.
pub struct Counter {
    ctx: *mut sys::DkbCtx,
    n_children: usize,
    n_entries: usize,
    n_variants: usize,
    /// region mode: copies of the loci of batches in flight (the library reads them until `sync`)
    loci_keep: Vec<[Vec<u64>; 3]>,
    _not_sync: PhantomData<*mut ()>,
}
unsafe impl Send for Counter {}

impl Counter {
    /// A trio context: child (sample 0), mother (1), father (2).
    pub fn new(device: i32, k: i32) -> Result<Self> {
        let mut ctx = ptr::null_mut();
        check(unsafe { sys::dkb_ctx_create(device, k, &mut ctx) }, ptr::null())?;
        Ok(Counter { ctx, n_children: 1, n_entries: 0, n_variants: 0, loci_keep: Vec::new(), _not_sync: PhantomData })
    }

    /// A family context: mother (sample 1), father (2) and `n_children` children (1..=6), child
    /// `c` being sample [`child_sample`]`(c)`, all counted against one table; the de novo rule
    /// is applied once per child.
    pub fn new_family(device: i32, k: i32, n_children: usize) -> Result<Self> {
        let mut ctx = ptr::null_mut();
        let n = c_int::try_from(n_children).unwrap_or(c_int::MAX);
        check(unsafe { sys::dkb_ctx_create_family(device, k, n, &mut ctx) }, ptr::null())?;
        Ok(Counter { ctx, n_children, n_entries: 0, n_variants: 0, loci_keep: Vec::new(), _not_sync: PhantomData })
    }

    pub fn n_children(&self) -> usize { self.n_children }
    /// 2 + n_children: the rows of the counters and the last axis of `hits` / `distinct`.
    pub fn n_samples(&self) -> usize { 2 + self.n_children }

    fn ck(&self, code: c_int) -> Result<()> { check(code, self.ctx) }

    pub fn set_tuning(&mut self, t: Option<Tuning>) -> Result<()> {
        self.ck(unsafe { sys::dkb_ctx_set_tuning(self.ctx, t.as_ref().map_or(ptr::null(), |t| t as *const _)) })
    }

    pub fn tuning(&self) -> Result<Tuning> {
        let mut t = Tuning::default();
        self.ck(unsafe { sys::dkb_ctx_get_tuning(self.ctx, &mut t) })?;
        Ok(t)
    }

    /// Kernel 1: build the spanning-k-mer table (replaces any previous table).
    pub fn build_table(&mut self, e: &Entries) -> Result<()> {
        let hints = e.win_index.len() == e.keys.len() && e.win_count.len() == e.keys.len();
        self.ck(unsafe {
            sys::dkb_table_build(self.ctx, e.keys.as_ptr(), e.variant.as_ptr(), e.allele.as_ptr(),
                                 if hints { e.win_index.as_ptr() } else { ptr::null() },
                                 if hints { e.win_count.as_ptr() } else { ptr::null() },
                                 e.keys.len(), e.n_variants)
        })?;
        self.n_entries = e.keys.len();
        self.n_variants = e.n_variants as usize;
        Ok(())
    }

    /// Kernel 2 on a packed batch held in a [`PinnedBatch`]: asynchronous H2D copy + scan.  The
    /// batch must not be repacked before [`Counter::sync`] (the packer's two-buffer rotation
    /// guarantees that when `sync` is called every second batch; see [`BatchPacker::next`]).
    pub fn submit(&mut self, b: &PinnedBatch, sample: i32) -> Result<()> {
        if b.zbytes_used != usize::MAX {
            // the packer made a zero list of the flags: a quarter less PCIe traffic
            return self.ck(unsafe {
                sys::dkb_batch_submit_sparse(self.ctx, b.bases2, b.zoff, b.zbytes, b.zbytes_used, b.n_positions, sample)
            });
        }
        self.ck(unsafe { sys::dkb_batch_submit(self.ctx, b.bases2, b.mask1, b.n_positions, sample) })
    }

    /// Kernel 2 on up to [`sys::DKB_MAX_MULTI`] packed batches, `(batch, sample)`, in ONE scan
    /// launch: a trio step is one call.  Each batch must not be repacked before
    /// [`Counter::sync`], as for [`Counter::submit`] (one [`BatchPacker`] per sample keeps that
    /// rule when `sync` is called every second step).  Region mode: [`Counter::set_loci_multi`] first.
    /// When every batch carries a zero list of its flags (as [`BatchPacker::next`] makes), the
    /// zero lists cross PCIe instead of the dense flags, as in [`Counter::submit`].
    pub fn submit_multi(&mut self, batches: &[(&PinnedBatch, i32)]) -> Result<()> {
        let b: Vec<*const u32> = batches.iter().map(|(x, _)| x.bases2 as *const u32).collect();
        let n: Vec<u64> = batches.iter().map(|(x, _)| x.n_positions).collect();
        let s: Vec<c_int> = batches.iter().map(|(_, smp)| *smp).collect();
        let nb = c_int::try_from(batches.len()).unwrap_or(c_int::MAX);
        if !batches.is_empty() && batches.iter().all(|(x, _)| x.zbytes_used != usize::MAX) {
            let z: Vec<*const u32> = batches.iter().map(|(x, _)| x.zoff as *const u32).collect();
            let zb: Vec<*const u8> = batches.iter().map(|(x, _)| x.zbytes as *const u8).collect();
            let used: Vec<usize> = batches.iter().map(|(x, _)| x.zbytes_used).collect();
            return self.ck(unsafe {
                sys::dkb_batch_submit_sparse_multi(self.ctx, nb, b.as_ptr(), z.as_ptr(), zb.as_ptr(), used.as_ptr(),
                                                   n.as_ptr(), s.as_ptr())
            });
        }
        let m: Vec<*const u32> = batches.iter().map(|(x, _)| x.mask1 as *const u32).collect();
        self.ck(unsafe { sys::dkb_batch_submit_multi(self.ctx, nb, b.as_ptr(), m.as_ptr(), n.as_ptr(), s.as_ptr()) })
    }

    /// Kernel 0 + 2: decoded reads as the BAM layer holds them (ASCII or 4-bit), packed on the GPU.
    pub fn submit_reads(&mut self, seq: &[u8], four_bit: bool, qual: Option<&[u8]>, offsets: &[u64],
                        min_baseq: i32, sample: i32) -> Result<()> {
        self.ck(unsafe {
            sys::dkb_batch_submit_reads(self.ctx, seq.as_ptr(), four_bit as c_int,
                                        qual.map_or(ptr::null(), |q| q.as_ptr()), offsets.as_ptr(),
                                        offsets.len().saturating_sub(1), min_baseq, sample)
        })
    }

    /// Kernel 0 + 2 on up to [`sys::DKB_MAX_MULTI`] batches of decoded reads,
    /// `(seq, qual, offsets, sample)`, packed in one launch and scanned in ONE: one `four_bit` and
    /// one `min_baseq` for all of them.  The buffers must stay unchanged until [`Counter::sync`].
    /// Region mode: [`Counter::set_loci_multi`] first.
    pub fn submit_reads_multi(&mut self, batches: &[(&[u8], Option<&[u8]>, &[u64], i32)], four_bit: bool,
                              min_baseq: i32) -> Result<()> {
        let seq: Vec<*const u8> = batches.iter().map(|b| b.0.as_ptr()).collect();
        let qual: Vec<*const u8> = batches.iter().map(|b| b.1.map_or(ptr::null(), |q| q.as_ptr())).collect();
        let off: Vec<*const u64> = batches.iter().map(|b| b.2.as_ptr()).collect();
        let nr: Vec<usize> = batches.iter().map(|b| b.2.len().saturating_sub(1)).collect();
        let s: Vec<c_int> = batches.iter().map(|b| b.3).collect();
        let nb = c_int::try_from(batches.len()).unwrap_or(c_int::MAX);
        self.ck(unsafe {
            sys::dkb_batch_submit_reads_multi(self.ctx, nb, seq.as_ptr(), four_bit as c_int, qual.as_ptr(),
                                              off.as_ptr(), nr.as_ptr(), min_baseq, s.as_ptr())
        })
    }

    /// Region mode (`include/dkb.h`): a read counts toward variant `v` only if its alignment
    /// interval overlaps `windows[v] = (lo, hi)`, half-open, one per variant of the table.  Every
    /// batch submitted after this needs its loci ([`Counter::set_loci`]).  A new table, or
    /// [`Counter::clear_regions`], returns to whole-stream counting.
    pub fn set_regions(&mut self, windows: &[(u64, u64)]) -> Result<()> {
        let lo: Vec<u64> = windows.iter().map(|w| w.0).collect();
        let hi: Vec<u64> = windows.iter().map(|w| w.1).collect();
        self.ck(unsafe { sys::dkb_table_set_regions(self.ctx, lo.as_ptr(), hi.as_ptr(), windows.len() as u32) })
    }

    pub fn clear_regions(&mut self) -> Result<()> {
        self.ck(unsafe { sys::dkb_table_set_regions(self.ctx, ptr::null(), ptr::null(), 0) })
    }

    /// Inheritance (`include/dkb.h`): the locus class of every variant of the table.  From now
    /// on each call applies only the clauses of the parents who can transmit the variant's locus
    /// to the child.  A new table, or [`Counter::clear_locus_classes`], returns to all autosomal.
    pub fn set_locus_classes(&mut self, cls: &[LocusClass]) -> Result<()> {
        let raw: Vec<u8> = cls.iter().map(|&c| c as u8).collect();
        let n = u32::try_from(raw.len()).unwrap_or(u32::MAX);
        self.ck(unsafe { sys::dkb_table_set_locus_classes(self.ctx, raw.as_ptr(), n) })
    }

    pub fn clear_locus_classes(&mut self) -> Result<()> {
        self.ck(unsafe { sys::dkb_table_set_locus_classes(self.ctx, ptr::null(), 0) })
    }

    /// Inheritance: the sex of every child, one per child of the context; kept across tables.
    pub fn set_child_sexes(&mut self, sexes: &[Sex]) -> Result<()> {
        let raw: Vec<u8> = sexes.iter().map(|&s| s as u8).collect();
        let n = c_int::try_from(raw.len()).unwrap_or(c_int::MAX);
        self.ck(unsafe { sys::dkb_ctx_set_child_sexes(self.ctx, raw.as_ptr(), n) })
    }

    /// Region mode: the loci of the NEXT submitted batch - the batch's `offsets` (as packed) and
    /// each read's alignment interval `[lo, hi)` (rust-htslib: `pos()`, `cigar().end_pos()`;
    /// `lo >= hi` for an unmapped read).  Copied here and kept until [`Counter::sync`].
    pub fn set_loci(&mut self, offsets: &[u64], lo: &[u64], hi: &[u64]) -> Result<()> {
        let keep = [offsets.to_vec(), lo.to_vec(), hi.to_vec()];
        let n_reads = offsets.len().saturating_sub(1);
        if lo.len() != n_reads || hi.len() != n_reads || offsets.is_empty() {
            return Err(DkbError { code: sys::DKB_EINVAL, detail: "lo and hi need one entry per read".into() });
        }
        self.ck(unsafe {
            sys::dkb_batch_set_loci(self.ctx, keep[0].as_ptr(), keep[1].as_ptr(), keep[2].as_ptr(), n_reads)
        })?;
        self.loci_keep.push(keep);  // (moving the Vecs does not move their heap buffers)
        Ok(())
    }

    /// Region mode: the loci of the NEXT multi-batch submit ([`Counter::submit_multi`]), one
    /// `(offsets, lo, hi)` per batch with the meaning of [`Counter::set_loci`].  Copied here and
    /// kept until [`Counter::sync`].
    pub fn set_loci_multi(&mut self, loci: &[(&[u64], &[u64], &[u64])]) -> Result<()> {
        let mut keep = Vec::with_capacity(loci.len());
        for (offsets, lo, hi) in loci {
            let n_reads = offsets.len().saturating_sub(1);
            if lo.len() != n_reads || hi.len() != n_reads || offsets.is_empty() {
                return Err(DkbError { code: sys::DKB_EINVAL, detail: "lo and hi need one entry per read".into() });
            }
            keep.push([offsets.to_vec(), lo.to_vec(), hi.to_vec()]);
        }
        let ptrs = |i: usize| keep.iter().map(|k| k[i].as_ptr()).collect::<Vec<*const u64>>();
        let (o, l, h) = (ptrs(0), ptrs(1), ptrs(2));
        let n: Vec<usize> = keep.iter().map(|k| k[1].len()).collect();
        let nb = c_int::try_from(loci.len()).unwrap_or(c_int::MAX);
        self.ck(unsafe { sys::dkb_batch_set_loci_multi(self.ctx, nb, o.as_ptr(), l.as_ptr(), h.as_ptr(), n.as_ptr()) })?;
        self.loci_keep.extend(keep);  // (moving the Vecs does not move their heap buffers)
        Ok(())
    }

    pub fn sync(&mut self) -> Result<()> {
        self.ck(unsafe { sys::dkb_sync(self.ctx) })?;
        self.loci_keep.clear();
        Ok(())
    }
    pub fn reset_counts(&mut self) -> Result<()> { self.ck(unsafe { sys::dkb_counts_reset(self.ctx) }) }

    /// Per-entry counts, `[n_samples][n_entries]`.
    pub fn entry_counts(&mut self) -> Result<Vec<u32>> {
        let mut out = vec![0u32; self.n_samples() * self.n_entries];
        self.ck(unsafe { sys::dkb_entry_counts_fetch(self.ctx, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// Kernel 3 + fetch.
    pub fn finalise(&mut self, thr: &Thresholds) -> Result<Results> {
        self.ck(unsafe { sys::dkb_finalise(self.ctx, thr) })?;
        self.results()
    }

    pub fn results(&mut self) -> Result<Results> {
        let (nv, ns) = (self.n_variants, self.n_samples());
        let mut r = Results { hits: vec![0; nv * 2 * ns], distinct: vec![0; nv * 2 * ns], n_kmers: vec![0; nv * 2],
                              calls: vec![0; nv * self.n_children] };
        self.ck(unsafe {
            sys::dkb_results_fetch(self.ctx, r.hits.as_mut_ptr(), r.distinct.as_mut_ptr(),
                                   r.n_kmers.as_mut_ptr(), r.calls.as_mut_ptr())
        })?;
        Ok(r)
    }

    pub fn stats(&mut self) -> Result<Stats> {
        let mut s = Stats::default();
        self.ck(unsafe { sys::dkb_stats_get(self.ctx, &mut s) })?;
        Ok(s)
    }

    // ---- multi-GPU -------------------------------------------------------------------------
    /// Join the communicator: `id` from [`comm_unique_id`] on rank 0, sent to every rank by the caller.
    pub fn comm_init(&mut self, id: &[u8; sys::DKB_COMM_ID_BYTES], rank: i32, world: i32) -> Result<()> {
        self.ck(unsafe { sys::dkb_comm_init(self.ctx, id.as_ptr() as *const c_void, rank, world) })
    }
    pub fn comm_destroy(&mut self) -> Result<()> { self.ck(unsafe { sys::dkb_comm_destroy(self.ctx) }) }
    /// In-place sum over ranks of the counters (then [`Counter::finalise`]).
    pub fn counts_allreduce(&mut self) -> Result<()> { self.ck(unsafe { sys::dkb_counts_allreduce(self.ctx) }) }
    /// Overlapped form: snapshot + sum on a side stream; finalises the previous snapshot.
    pub fn reduce_push(&mut self, thr: &Thresholds) -> Result<()> { self.ck(unsafe { sys::dkb_reduce_push(self.ctx, thr) }) }
    pub fn reduce_flush(&mut self, thr: &Thresholds) -> Result<()> { self.ck(unsafe { sys::dkb_reduce_flush(self.ctx, thr) }) }
    pub fn reduced_counts(&mut self) -> Result<Vec<u32>> {
        let mut out = vec![0u32; self.n_samples() * self.n_entries];
        self.ck(unsafe { sys::dkb_reduced_counts_fetch(self.ctx, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// Pin the calling thread to the CPUs next to this GPU; returns the NUMA node (-1 unknown).
    pub fn bind_thread_near_gpu(&mut self) -> Result<i32> {
        let mut node: c_int = -1;
        self.ck(unsafe { sys::dkb_thread_bind_near_gpu(self.ctx, &mut node) })?;
        Ok(node)
    }

    /// Two page-locked batch buffers next to this GPU, each for up to `max_bases` read bases in
    /// `max_reads` reads.
    pub fn batch_packer(&mut self, max_reads: usize, max_bases: usize, min_baseq: i32) -> Result<BatchPacker> {
        BatchPacker::new(self, max_reads, max_bases, min_baseq)
    }
}

impl Drop for Counter {
    fn drop(&mut self) {
        unsafe { sys::dkb_ctx_destroy(self.ctx) };
    }
}

/// Rank 0: the NCCL id every rank passes to [`Counter::comm_init`].
pub fn comm_unique_id() -> Result<[u8; sys::DKB_COMM_ID_BYTES]> {
    let mut id = [0u8; sys::DKB_COMM_ID_BYTES];
    check(unsafe { sys::dkb_comm_unique_id(id.as_mut_ptr() as *mut c_void) }, ptr::null())?;
    Ok(id)
}

/// One packed batch in page-locked memory (owned by its [`BatchPacker`]).
pub struct PinnedBatch {
    bases2: *mut u32,
    mask1: *mut u32,
    zoff: *mut u32,   // the flags as a zero list (dkb_mask_to_zero_list), also pinned
    zbytes: *mut u8,
    zbytes_cap: usize,
    zbytes_used: usize, // usize::MAX: no zero list, submit the dense flags
    cap_bw: usize,
    cap_mw: usize,
    pub n_positions: u64,
    pub n_bases: u64,
}

/// Packs decoded reads into two rotating pinned buffers.
pub struct BatchPacker {
    ctx: *mut sys::DkbCtx,
    bufs: [PinnedBatch; 2],
    next: usize,
    min_baseq: i32,
}

impl BatchPacker {
    fn new(c: &mut Counter, max_reads: usize, max_bases: usize, min_baseq: i32) -> Result<Self> {
        let n_pos = (max_bases + max_reads) as u64;
        let (bw, mw) = unsafe { (sys::dkb_stream_bases_words(n_pos), sys::dkb_stream_mask_words(n_pos)) };
        let nb = unsafe { sys::dkb_zero_list_blocks(n_pos) };
        let zcap = mw * 4; // a zero list is never longer than the dense flags
        let mut mk = || -> Result<PinnedBatch> {
            let (mut b, mut m, mut zo, mut zb) = (ptr::null_mut(), ptr::null_mut(), ptr::null_mut(), ptr::null_mut());
            check(unsafe { sys::dkb_host_alloc(c.ctx, bw * 4, &mut b) }, c.ctx)?;
            check(unsafe { sys::dkb_host_alloc(c.ctx, mw * 4, &mut m) }, c.ctx)?;
            check(unsafe { sys::dkb_host_alloc(c.ctx, (nb + 1) * 4, &mut zo) }, c.ctx)?;
            check(unsafe { sys::dkb_host_alloc(c.ctx, zcap, &mut zb) }, c.ctx)?;
            Ok(PinnedBatch { bases2: b as *mut u32, mask1: m as *mut u32, zoff: zo as *mut u32,
                             zbytes: zb as *mut u8, zbytes_cap: zcap, zbytes_used: usize::MAX,
                             cap_bw: bw, cap_mw: mw, n_positions: 0, n_bases: 0 })
        };
        Ok(BatchPacker { ctx: c.ctx, bufs: [mk()?, mk()?], next: 0, min_baseq })
    }

    /// `dkb_pack_reads_fmt` into the next buffer: `seq`/`qual` are the reads back to back, read r at
    /// `offsets[r]..offsets[r + 1]` (in bases).  `four_bit`: `seq` holds BAM 4-bit codes
    /// (`record.seq().encoded`, every read on a byte boundary) instead of ASCII - no decode pass.
    /// The buffer returned was last handed out two calls ago: call [`Counter::sync`] at least
    /// every second batch before packing again.
    pub fn next(&mut self, seq: &[u8], four_bit: bool, qual: Option<&[u8]>, offsets: &[u64]) -> Result<&PinnedBatch> {
        let n_reads = offsets.len().saturating_sub(1);
        let n_pos = unsafe { sys::dkb_stream_positions(offsets.as_ptr(), n_reads) };
        let b = &mut self.bufs[self.next];
        self.next ^= 1;
        let (bw, mw) = unsafe { (sys::dkb_stream_bases_words(n_pos), sys::dkb_stream_mask_words(n_pos)) };
        if bw > b.cap_bw || mw > b.cap_mw {
            return Err(DkbError { code: sys::DKB_EINVAL, detail: "batch larger than the packer's buffers".into() });
        }
        let mut out = 0u64;
        check(unsafe {
            sys::dkb_pack_reads_fmt(seq.as_ptr(), four_bit as c_int, qual.map_or(ptr::null(), |q| q.as_ptr()),
                                    offsets.as_ptr(), n_reads, self.min_baseq, b.bases2, b.mask1, &mut out)
        }, self.ctx)?;
        b.n_positions = out;
        b.n_bases = if n_reads > 0 { offsets[n_reads] - offsets[0] } else { 0 };
        let mut used = 0usize;
        check(unsafe {
            sys::dkb_mask_to_zero_list(b.mask1, out, b.zoff, b.zbytes, b.zbytes_cap, &mut used)
        }, self.ctx)?;
        b.zbytes_used = used;
        Ok(b)
    }
}

impl Drop for BatchPacker {
    fn drop(&mut self) {
        // the context outlives its packers in correct use; freeing pinned memory needs no context
        for b in &self.bufs {
            unsafe {
                sys::dkb_host_free(ptr::null_mut(), b.bases2 as *mut c_void);
                sys::dkb_host_free(ptr::null_mut(), b.mask1 as *mut c_void);
                sys::dkb_host_free(ptr::null_mut(), b.zoff as *mut c_void);
                sys::dkb_host_free(ptr::null_mut(), b.zbytes as *mut c_void);
            }
        }
    }
}

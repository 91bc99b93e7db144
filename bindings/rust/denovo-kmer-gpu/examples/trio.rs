//! The loop INTEGRATION.md §3 describes, as code: what the reference's `main.rs` does around
//! `kmer.rs` / `counter.rs`, with the GPU counter in their place.  The BAM / VCF / FASTA side is
//! the reference's own (rust-htslib) and is represented here by the `ReadSource` trait.
use denovo_kmer_gpu::{child_sample, comm_unique_id, variant_kmers, Candidate, Counter, Thresholds, CALL_DENOVO};

/// What the reference's BAM layer yields: decoded reads of one sample, in batches.
pub trait ReadSource {
    /// Fills `seq` (ASCII here; `record.seq().encoded` with `four_bit = true` skips the decode),
    /// `qual`, `offsets` (offsets[0] = 0) with the next batch; false at end of file.
    fn next_batch(&mut self, seq: &mut Vec<u8>, qual: &mut Vec<u8>, offsets: &mut Vec<u64>) -> bool;
    /// The alignment intervals of the last batch's reads in the linear coordinates of
    /// `cand_pos` (contig offset + `record.pos()` .. `record.cigar().end_pos()`; `lo >= hi` for
    /// an unmapped read).  Needed in region mode only.
    fn loci(&self, lo: &mut Vec<u64>, hi: &mut Vec<u64>);
}

/// Region mode: count a read toward a candidate only if it aligned within `window` bases of it
/// (what fetching reads per candidate window does).  `cand_pos`: each candidate's position in the
/// same linear coordinates as `ReadSource::loci`.
pub struct Regions<'a> {
    pub cand_pos: &'a [u64],
    pub window: u64,
}

/// `samples`: child, mother, father.  `second_child`: a quad - one family context counts both
/// children against one table, and each parent's BAM is read once (the second child is
/// sample `child_sample(1)` = 3).  `one_launch`: read one batch of every sample per step and
/// scan the step's batches in ONE launch (`submit_multi`) - worth it when batches are small, as
/// when reads are fetched per candidate window.  Returns the de novo calls per child, then per
/// candidate.
pub fn run_trio(device: i32, k: i32, min_baseq: i32, thr: Thresholds, cands: &[Candidate<'_>],
                samples: &mut [Box<dyn ReadSource>; 3], second_child: Option<Box<dyn ReadSource>>,
                rank_world: Option<(i32, i32, [u8; 128])>,
                regions: Option<Regions<'_>>, one_launch: bool) -> denovo_kmer_gpu::Result<Vec<Vec<bool>>> {
    let n_children = if second_child.is_some() { 2 } else { 1 };
    let mut kc = Counter::new_family(device, k, n_children)?;
    kc.bind_thread_near_gpu()?;
    if let Some((rank, world, id)) = rank_world {
        kc.comm_init(&id, rank, world)?; // every rank scans its own slice of the read batches
    }
    kc.build_table(&variant_kmers(cands, k, true)?)?;
    if let Some(r) = &regions {
        let w: Vec<(u64, u64)> =
            r.cand_pos.iter().map(|&p| (p.saturating_sub(r.window), p.saturating_add(r.window + 1))).collect();
        kc.set_regions(&w)?;
    }
    let (mut lo, mut hi) = (Vec::new(), Vec::new());
    let mut packer = kc.batch_packer(1 << 21, 150 << 21, min_baseq)?;
    let (mut seq, mut qual, mut off) = (Vec::new(), Vec::new(), Vec::new());
    let mut second = second_child.into_iter().map(|src| (child_sample(1), src)).collect::<Vec<_>>();
    let sources = samples.iter_mut().enumerate().chain(second.iter_mut().map(|(s, src)| (*s, src)));
    if one_launch {
        // one packer (two pinned buffers) and one batch per sample and step
        let mut srcs: Vec<(usize, &mut Box<dyn ReadSource>)> = sources.collect();
        let mut packers = Vec::new();
        for _ in 0..srcs.len() {
            packers.push(kc.batch_packer(1 << 21, 150 << 21, min_baseq)?);
        }
        let mut bufs = vec![(Vec::new(), Vec::new(), Vec::new(), Vec::new(), Vec::new()); srcs.len()];
        let (mut live, mut in_flight) = (vec![true; srcs.len()], 0);
        while live.iter().any(|&l| l) {
            if in_flight == 2 {
                kc.sync()?; // every packer's two buffers are in use
                in_flight = 0;
            }
            for (i, (_, src)) in srcs.iter_mut().enumerate() {
                let (seq, qual, off, lo, hi) = &mut bufs[i];
                live[i] = live[i] && src.next_batch(seq, qual, off);
                if live[i] && regions.is_some() {
                    src.loci(lo, hi);
                }
            }
            let step: Vec<usize> = (0..srcs.len()).filter(|&i| live[i]).collect();
            if regions.is_some() {
                let loci: Vec<(&[u64], &[u64], &[u64])> =
                    step.iter().map(|&i| (bufs[i].2.as_slice(), bufs[i].3.as_slice(), bufs[i].4.as_slice())).collect();
                kc.set_loci_multi(&loci)?;
            }
            let mut batches = Vec::new();
            for (i, p) in packers.iter_mut().enumerate().filter(|(i, _)| live[*i]) {
                let (seq, qual, off, _, _) = &bufs[i];
                batches.push((p.next(seq, false, Some(qual.as_slice()), off)?, srcs[i].0 as i32));
            }
            // the packers made zero lists of the flags, so this one launch also sends the smaller
            // zero lists over PCIe (dkb_batch_submit_sparse_multi), as `submit` does below
            kc.submit_multi(&batches)?;
            in_flight += 1;
        }
        kc.sync()?;
    } else {
        for (sample, src) in sources {
            let mut in_flight = 0;
            while src.next_batch(&mut seq, &mut qual, &mut off) {
                if in_flight == 2 {
                    kc.sync()?; // both pinned buffers are in use: wait before repacking one
                    in_flight = 0;
                }
                if regions.is_some() {
                    src.loci(&mut lo, &mut hi);
                    kc.set_loci(&off, &lo, &hi)?;
                }
                let batch = packer.next(&seq, false, Some(qual.as_slice()), &off)?;
                kc.submit(batch, sample as i32)?;
                in_flight += 1;
            }
            kc.sync()?;
        }
    }
    kc.counts_allreduce()?; // no-op without a communicator
    let res = kc.finalise(&thr)?;
    // calls[v * n_children + c]: child c's byte for candidate v
    Ok((0..n_children)
        .map(|c| res.calls.iter().skip(c).step_by(n_children).map(|b| b & CALL_DENOVO != 0).collect())
        .collect())
}

fn main() {
    // rank 0 of a multi-GPU job would make the id and send it round:
    let _ = comm_unique_id();
    eprintln!("see run_trio(); the reference's CLI supplies the candidates and the three (or four) BAM readers");
}

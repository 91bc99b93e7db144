"""CPU reference for family contexts, composed from the unchanged trio oracle (oracle/):
every sample is counted with KmerSet.count_reads, and child c's per-variant statistics and
calls come from variant_stats and calls on the trio of rows [child_sample(c), 1, 2]."""
import numpy as np

from denovo_kmer_b200.synth import child_sample


def family_counts(orc, entries, fam, k, min_bq, n_samples):
    """(KmerSet, uint64 [n_samples, n_entries]) from each sample's reads in fam.reads."""
    ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
    counts = np.zeros((n_samples, len(entries)), dtype=np.uint64)
    for smp in range(n_samples):
        seq, qual, off = fam.reads[smp]
        ks.count_reads(seq, qual, off, k, min_bq, counts=counts[smp])
    return ks, counts


def family_results(orc, ks, counts, n_variants, n_children, thr):
    """hits, distinct [nv, 2, NS], n_kmers [nv, 2] and calls [nv, n_children] of the counters."""
    ns = 2 + n_children
    hits = np.zeros((n_variants, 2, ns), dtype=np.uint64)
    dist = np.zeros((n_variants, 2, ns), dtype=np.uint64)
    calls = np.zeros((n_variants, n_children), dtype=np.uint8)
    nk = None
    for c in range(n_children):
        rows = [child_sample(c), 1, 2]
        h, d, nk = ks.variant_stats(counts[rows], n_variants)
        hits[:, :, rows] = h
        dist[:, :, rows] = d
        calls[:, c] = orc.calls(h, d, thr)
    return hits, dist, nk, calls

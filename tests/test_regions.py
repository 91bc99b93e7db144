"""CPU: region-scoped counting's references and host-side pieces.  The C stream walk with read
loci equals a per-variant read fetch in plain Python, reduces to the whole-stream oracle when
every window covers every read, and gives zeros when they all miss; synth's read loci are
where the reads came from; the paralog plant puts ALT copies far from every candidate; the
bindings declare the two new entry points."""
import os
import re

import numpy as np
import pytest

import region_oracle as ro
from denovo_kmer_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _entries(orc, trio, k, drop_shared=True):
    keys, var, al, _, _ = orc.variant_entries(trio.variant_tuples(), k, drop_shared)
    return keys, var, al


def _stream_loci(orc, trio, k, keys, var, al, vlo, vhi, min_bq):
    out = np.zeros((3, len(keys)), dtype=np.uint64)
    for smp in range(3):
        seq, qual, off = trio.reads[smp]
        b2, m1, n_pos = orc.pack_stream(seq, qual, off, min_bq)
        lo, hi = trio.loci[smp]
        ro.count_stream_loci(keys, var, al, vlo, vhi, b2, m1, n_pos, off, lo, hi, k, counts=out[smp])
    return out


@pytest.mark.parametrize("k,indel_frac,drop_shared,pad", [(21, 0.0, True, 40), (31, 0.5, True, 200),
                                                          (31, 0.5, False, 0), (15, 0.3, True, 1000)])
def test_loci_oracle_equals_per_variant_fetch(orc, k, indel_frac, drop_shared, pad):
    trio = synth.make_trio_host(12_000, 8, 6, k, seed=40 + k, indel_frac=indel_frac, ragged=True,
                                n_rate=0.005, lowq_frac=0.05)
    keys, var, al = _entries(orc, trio, k, drop_shared)
    vlo, vhi = ro.windows(trio.variants, pad)
    vhi[1] = vlo[1]  # an empty window: nothing counts toward variant 1
    for smp in range(3):  # a few unmapped reads
        lo, hi = trio.loci[smp]
        hi[::17] = lo[::17]
    got = _stream_loci(orc, trio, k, keys, var, al, vlo, vhi, 20)
    want = ro.py_fetch_counts(keys, var, al, len(trio.variants), vlo, vhi,
                              [ro.trio_reads(trio, s) for s in range(3)], k, 20)
    assert np.array_equal(got, want)
    assert got.sum() > 0 and got[:, var == 1].sum() == 0


def test_loci_oracle_reduces_to_whole_stream(orc):
    k = 31
    trio = synth.make_trio_host(30_000, 10, 10, k, seed=9, indel_frac=0.4)
    keys, var, al = _entries(orc, trio, k)
    nv = len(trio.variants)
    ks = orc.KmerSet(keys, var, al)
    whole = np.zeros((3, len(keys)), dtype=np.uint64)
    for smp in range(3):
        ks.count_stream(*orc.pack_stream(*trio.reads[smp], 20), k, counts=whole[smp])
    cover = _stream_loci(orc, trio, k, keys, var, al, np.zeros(nv, np.uint64), np.full(nv, 1 << 40, np.uint64), 20)
    assert np.array_equal(cover, whole) and whole.sum() > 0
    miss = _stream_loci(orc, trio, k, keys, var, al, np.full(nv, 1 << 40, np.uint64),
                        np.full(nv, (1 << 40) + 5, np.uint64), 20)
    assert miss.sum() == 0


def test_synth_read_loci_are_true_alignments():
    """Error-free reads: a read that overlaps no variant equals the genome on [lo, hi) (or its
    reverse complement); reads over an insertion span fewer genome bases, over a deletion more."""
    trio = synth.make_trio_host(40_000, 6, 12, 31, seed=21, indel_frac=0.6, ragged=True,
                                err_rate=0.0, n_rate=0.0)
    g = trio.genome
    comp = synth.COMP_ASCII
    for smp in range(3):
        seq, _, off = trio.reads[smp]
        lo, hi = trio.loci[smp]
        assert len(lo) == len(off) - 1 and (hi >= lo).all() and (hi <= len(g)).all()
        for r in range(0, len(lo), 7):
            s = seq[int(off[r]):int(off[r + 1])]
            a, b = int(lo[r]), int(hi[r])
            hit = [v for v in trio.variants if v.pos < b and a < v.pos + len(v.ref)]
            if not hit:
                assert np.array_equal(s, g[a:b]) or np.array_equal(s, comp[g[a:b][::-1]]), (smp, r)
    # the father carries no variant: every read is a plain genome interval of its own length
    _, _, off = trio.reads[2]
    lo, hi = trio.loci[2]
    assert np.array_equal((hi - lo).astype(np.int64), np.diff(off).astype(np.int64))


def test_paralog_plant():
    k = 31
    trio = synth.make_trio_host(60_000, 4, 12, k, seed=5, paralog_frac=0.5)
    assert trio.paralogs and all(not trio.variants[i].inherited for i in trio.paralogs)
    g = trio.genome.tobytes()
    last = max(v.pos for v in trio.variants)
    for i in trio.paralogs:
        left, ref, alt, right = trio.variant_tuples()[i]
        copy = (left + alt + right).encode()
        at = g.find(copy)
        assert at > last + 10_000, (i, at)  # far from every candidate window
    # the father's reads reach the copies
    assert int(trio.loci[2][1].max()) > 60_000


def test_device_read_loci_cpu():
    """make_sample_device's return_meta starts as loci (CPU torch): a genome-only sample's reads
    span read_len genome bases from where they were drawn."""
    torch = pytest.importorskip("torch")
    genome = synth.make_genome(20_000, 1)
    lut = np.zeros(256, dtype=np.uint8)
    for i, ch in enumerate(b"ACGT"):
        lut[ch] = i
    g = torch.from_numpy(lut[genome])
    variants = synth.plant_variants(genome, 5, 31, 2, indel_frac=0.6)
    alt = torch.from_numpy(lut[synth.apply_variants(genome, variants)])
    *_, meta = synth.make_sample_device([g, alt], 256, 150, 3, torch.device("cpu"), chunk_reads=128,
                                        return_meta=True)
    off, lo, hi = synth.device_read_loci(meta, [None, synth.hap_ref_positions(genome, variants)], 150)
    assert len(off) == 257 and off[-1] == 256 * 150
    from_genome = meta[0].numpy() == 0
    assert (hi - lo)[from_genome].tolist() == [150] * int(from_genome.sum())
    assert (hi > lo).all() and (hi <= len(genome)).all()


def test_bindings_declare_region_mode(dkb):
    from denovo_kmer_b200 import _lib
    for name in ("dkb_table_set_regions", "dkb_batch_set_loci"):
        assert name in _lib.SYMBOLS
        assert hasattr(_lib.lib(), name)
    for m in ("set_regions", "clear_regions"):
        assert hasattr(dkb.KmerCounter, m)
    for m in ("submit", "submit_sparse", "submit_reads", "submit_device"):
        assert "loci" in getattr(dkb.KmerCounter, m).__code__.co_varnames
    with pytest.raises(ValueError):
        dkb.ReadLoci(np.array([0, 5, 9]), np.array([1]), np.array([2]))
    hpp = open(os.path.join(ROOT, "include", "dkb.hpp")).read()
    assert "dkb_table_set_regions" in hpp and "dkb_batch_set_loci" in hpp
    safe = open(os.path.join(ROOT, "bindings", "rust", "denovo-kmer-gpu", "src", "lib.rs")).read()
    assert re.search(r"pub fn set_regions\(&mut self, windows: &\[\(u64, u64\)\]\)", safe)
    assert "pub fn set_loci" in safe
    example = open(os.path.join(ROOT, "bindings", "rust", "denovo-kmer-gpu", "examples", "trio.rs")).read()
    assert "kc.set_regions(" in example and "kc.set_loci(" in example

"""CPU: family contexts without a GPU - the synthetic family generator, the family oracle
composed from the trio oracle (tests/family_oracle.py) on a small quad with a known answer,
the unchanged trio generator, and the ABI's family refusals that come before the device."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from denovo_kmer_b200 import synth
from family_oracle import family_counts, family_results

K = 31
THR = (3, 2, 0, 1)
CALL_DENOVO, CALL_CHILD_LOW, CALL_MOTHER_ALT, CALL_FATHER_ALT = 0x01, 0x02, 0x04, 0x08
CLEAN = dict(err_rate=0.0, n_rate=0.0, lowq_frac=0.0)


def _alt_hits(orc, dkb, fam, min_bq=0):
    """alt k-mer hits [nv, NS] of every sample, from the oracle on the family's reads."""
    ns = 2 + fam.n_children
    entries = dkb.variant_kmers(fam.variant_tuples(), K)
    ks, counts = family_counts(orc, entries, fam, K, min_bq, ns)
    out = np.zeros((len(fam.variants), ns), dtype=np.uint64)
    alt = entries.allele == 1
    for smp in range(ns):
        np.add.at(out[:, smp], entries.variant[alt], counts[smp][alt])
    return out


def _trio_hash(t):
    m = hashlib.sha256()
    m.update(t.genome.tobytes())
    for v in t.variants:
        m.update(repr((v.pos, v.ref, v.alt, v.inherited)).encode())
    for s in sorted(t.reads):
        for a in t.reads[s] + t.loci[s]:
            m.update(np.ascontiguousarray(a).tobytes())
    m.update(repr(t.paralogs).encode())
    return m.hexdigest()


def test_trio_generator_unchanged():
    """make_trio_host returns what it returned before families existed (hashes taken then)."""
    t = synth.make_trio_host(60_000, 6, 12, K, seed=4, indel_frac=0.4)
    assert _trio_hash(t) == "9f90d6792e1c330b83ad231447d6f1493817b15be1ff44e2c324480b690eea6a"
    t = synth.make_trio_host(60_000, 6, 12, K, seed=9, ragged=True, paralog_frac=0.3)
    assert _trio_hash(t) == "ca11b2687245ced746f90e9c814156a2b0ea9e01747e9a14de4584e4961c90e1"
    assert all(v.owner == 0 and v.carriers == {0} for v in t.variants) and t.n_children == 1


@pytest.mark.parametrize("n_children", [1, 2, 3, 6])
def test_family_generator_structure(n_children):
    fam = synth.make_family_host(150_000, 4, 36, K, n_children, seed=21, indel_frac=0.3,
                                 shared_frac=0.3, inherited_frac=0.3, ragged=True)
    ns = 2 + n_children
    assert sorted(fam.reads) == sorted(fam.loci) == list(range(ns)) and fam.n_children == n_children
    kinds = set()
    for i, v in enumerate(fam.variants):
        assert v.owner == i % n_children
        assert v.carriers <= set(range(n_children))
        if v.inherited:
            kinds.add("inherited")
        elif len(v.carriers) == 2:
            kinds.add("shared")
            assert v.owner in v.carriers and n_children > 1
        else:
            kinds.add("denovo")
            assert v.carriers == {v.owner}
    assert kinds == ({"denovo", "shared", "inherited"} if n_children > 1 else {"denovo", "inherited"})
    for smp in range(ns):
        seq, qual, off = fam.reads[smp]
        lo, hi = fam.loci[smp]
        assert len(lo) == len(hi) == len(off) - 1 and len(seq) == len(qual) == off[-1]
        assert (lo <= hi).all() and (hi <= len(fam.genome)).all()
        assert (hi > lo)[np.diff(off) > 0].all()


@pytest.mark.parametrize("n_children", [2, 3])
def test_family_generator_haplotypes(dkb, orc, n_children):
    """From error-free reads: each child's alt haplotype holds exactly the variants it carries
    (its reads hold their alt k-mers, and no others'), the mother exactly the inherited ones,
    the father none."""
    fam = synth.make_family_host(120_000, 24, 24, K, n_children, seed=31, indel_frac=0.3,
                                 shared_frac=0.3, inherited_frac=0.3, **CLEAN)
    alt = _alt_hits(orc, dkb, fam)
    for i, v in enumerate(fam.variants):
        for c in range(n_children):
            assert (alt[i, synth.child_sample(c)] > 0) == (c in v.carriers), (i, c, v)
        assert (alt[i, 1] > 0) == v.inherited, (i, v)
        assert alt[i, 2] == 0, (i, v)


def test_family_oracle_known_answer_quad(dkb, orc):
    """A quad (two children) with every kind of variant: the per-child calls of the oracle
    composed from the trio oracle."""
    fam = synth.make_family_host(200_000, 24, 40, K, 2, seed=41, shared_frac=0.3, inherited_frac=0.3, **CLEAN)
    entries = dkb.variant_kmers(fam.variant_tuples(), K)
    ks, counts = family_counts(orc, entries, fam, K, 0, 4)
    hits, dist, nk, calls = family_results(orc, ks, counts, len(fam.variants), 2, THR)
    assert calls.shape == (len(fam.variants), 2) and hits.shape == (len(fam.variants), 2, 4)
    seen = set()
    for i, v in enumerate(fam.variants):
        if v.inherited:
            seen.add("inherited")
            for c in range(2):
                assert not calls[i, c] & CALL_DENOVO and calls[i, c] & CALL_MOTHER_ALT, (i, c)
                assert bool(calls[i, c] & CALL_CHILD_LOW) == (c not in v.carriers), (i, c)
        elif len(v.carriers) == 2:
            seen.add("shared")
            assert calls[i].tolist() == [CALL_DENOVO, CALL_DENOVO], i
        else:
            seen.add("denovo")
            assert calls[i, v.owner] == CALL_DENOVO, i
            assert calls[i, 1 - v.owner] == CALL_CHILD_LOW, i
    assert seen == {"denovo", "shared", "inherited"}
    # child c's columns are the trio statistics of rows [child_sample(c), 1, 2]
    for c in range(2):
        rows = [synth.child_sample(c), 1, 2]
        h, d, n = ks.variant_stats(counts[rows], len(fam.variants))
        assert np.array_equal(hits[:, :, rows], h) and np.array_equal(dist[:, :, rows], d)
        assert np.array_equal(nk, n)


def test_create_family_refusals_before_device(dkb):
    from denovo_kmer_b200 import _lib
    L = _lib.lib()
    h = C.c_void_p()
    for n in (0, 7, -1):
        assert L.dkb_ctx_create_family(0, 31, n, C.byref(h)) == _lib.EINVAL
        assert not h.value
        with pytest.raises(dkb.DkbError) as ei:
            dkb.KmerCounter(31, n_children=n)
        assert ei.value.code == _lib.EINVAL
    assert L.dkb_ctx_create_family(0, 7, 2, C.byref(h)) == _lib.EINVAL  # k is checked first too
    assert L.dkb_ctx_get_children(None, None) == _lib.EINVAL
    assert [dkb.KmerCounter.child_sample(c) for c in range(6)] == [0, 3, 4, 5, 6, 7]


def test_create_family_without_gpu(dkb):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from denovo_kmer_b200 import _lib
    h = C.c_void_p()
    assert _lib.lib().dkb_ctx_create_family(0, 31, 2, C.byref(h)) == _lib.ENODEV
    with pytest.raises(dkb.DkbError) as ei:
        dkb.KmerCounter(31, n_children=2)
    assert ei.value.code == _lib.ENODEV


def test_bindings_declare_family_mode():
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "dkb.h")).read()
    assert "#define DKB_MAX_CHILDREN 6" in hdr
    sysrs = open(os.path.join(root, "bindings", "rust", "denovo-kmer-gpu-sys", "src", "lib.rs")).read()
    assert "pub const DKB_MAX_CHILDREN: usize = 6;" in sysrs
    safe = open(os.path.join(root, "bindings", "rust", "denovo-kmer-gpu", "src", "lib.rs")).read()
    assert re.search(r"pub fn new_family\(device: i32, k: i32, n_children: usize\)", safe)
    example = open(os.path.join(root, "bindings", "rust", "denovo-kmer-gpu", "examples", "trio.rs")).read()
    assert "Counter::new_family(" in example and "child_sample(1)" in example
    hpp = open(os.path.join(root, "include", "dkb.hpp")).read()
    assert "dkb_ctx_create_family(device, k, n_children, &ctx_)" in hpp

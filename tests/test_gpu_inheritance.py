"""-m gpu: kernel 3 with locus classes and child sexes (include/dkb.h "inheritance") against the
inheritance oracle (tests/inherit_oracle.py): crafted counters through dkb_finalise_from for
one, two and six children, the sexed family generator end to end (whole-stream and region
mode), the overlapped reduction recording classes and sexes with each snapshot, and the
refusals."""
import numpy as np
import pytest
import torch

import inherit_oracle as io
import region_oracle as ro
from denovo_kmer_b200 import synth
from family_oracle import family_counts

pytestmark = pytest.mark.gpu

K, THR, MIN_BQ = 31, (3, 2, 0, 1), 20
M, F, U = synth.SEX_MALE, synth.SEX_FEMALE, synth.SEX_UNKNOWN
A, X, Y, MT = synth.LOCUS_AUTOSOMAL, synth.LOCUS_X, synth.LOCUS_Y, synth.LOCUS_MATERNAL
# which parents' clauses apply (DESIGN.md §2); "-": neither, and the child has no copy
TABLE = {(A, U): "MF", (A, M): "MF", (A, F): "MF", (X, U): "MF", (X, M): "M", (X, F): "MF",
         (Y, U): "MF", (Y, M): "F", (Y, F): "-", (MT, U): "M", (MT, M): "M", (MT, F): "M"}


def _entries(dkb, nv, per_allele=2):
    """per_allele distinct keys for each allele of each of nv variants (no window hints)."""
    n = nv * 2 * per_allele
    keys = (np.arange(n, dtype=np.uint64) * np.uint64(7919) + np.uint64(12345))
    var = np.repeat(np.arange(nv, dtype=np.uint32), 2 * per_allele)
    al = np.tile(np.repeat(np.array([0, 1], np.uint8), per_allele), nv)
    return dkb.KmerEntries(keys, var, al, None, None, nv)


@pytest.mark.parametrize("n_children,sexes", [(1, [U]), (1, [M]), (1, [F]), (2, [M, F]), (6, [U, M, F, F, M, U])])
def test_crafted_counters(dkb, orc, n_children, sexes):
    """Random small counters cover every (class, sex) cell and clause; hits / distinct /
    n_kmers stay exact, calls equal the oracle's with classes and sexes, and today's without."""
    nv = 6000
    rng = np.random.default_rng(n_children * 10 + sexes[0])
    entries = _entries(dkb, nv)
    ns = 2 + n_children
    counts = rng.integers(0, 4, size=(ns, len(entries))).astype(np.uint32)
    counts[rng.random(counts.shape) < 0.3] = 0
    classes = rng.integers(0, 4, size=nv).astype(np.uint8)
    ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
    c64 = counts.astype(np.uint64)
    want = io.family_results(orc, ks, c64, nv, n_children, THR, classes, sexes)
    plain = io.family_results(orc, ks, c64, nv, n_children, THR)
    thr2 = (2, 1, 1, 2)
    want2 = io.family_results(orc, ks, c64, nv, n_children, thr2, classes, sexes)
    d_counts = torch.from_numpy(counts.view(np.int32).copy()).cuda()
    torch.cuda.synchronize()
    with dkb.KmerCounter(K, n_children=n_children) as kc:
        kc.build_table(entries, use_window_hints=False)
        kc.set_locus_classes(classes)
        kc.set_child_sexes(sexes)
        got = []
        for thr in (THR, thr2):
            kc.finalise_launch(thr, counts_ptr=d_counts.data_ptr())
            got.append(tuple(x.copy() for x in kc.results()))
        kc.clear_locus_classes()
        kc.set_child_sexes(None)
        kc.finalise_launch(THR, counts_ptr=d_counts.data_ptr())
        got_plain = tuple(x.copy() for x in kc.results())
    for (hits, dist, nk, calls), w in ((got[0], want), (got[1], want2), (got_plain, plain)):
        assert np.array_equal(hits.astype(np.uint64), w[0]) and np.array_equal(dist.astype(np.uint64), w[1])
        assert np.array_equal(nk, w[2])
        assert np.array_equal(calls.reshape(nv, n_children), w[3])
    # every cell of the table shows exactly the clause bits of the parents it names
    calls = got[0][3].reshape(nv, n_children)
    for c, sex in enumerate(sexes):
        for cls in range(4):
            who = TABLE[(cls, sex)]
            sel = calls[classes == cls, c]
            bits = int(np.bitwise_or.reduce(sel))
            want_bits = 0x02 | (0x04 if "M" in who else 0) | (0x08 if "F" in who else 0)
            want_bits |= 0x20 if who == "-" else 0x11
            assert bits == want_bits, (cls, sex, hex(bits))
    assert not np.array_equal(calls, got_plain[3].reshape(nv, n_children))


def _fam_oracle(dkb, orc, fam, region):
    entries = dkb.variant_kmers(fam.variant_tuples(), K)
    ns = 2 + fam.n_children
    if region:
        vlo, vhi = ro.windows(fam.variants, 400)
        want = np.zeros((ns, len(entries)), dtype=np.uint64)
        for smp in range(ns):
            seq, qual, off = fam.reads[smp]
            b2, m1, n_pos = orc.pack_stream(seq, qual, off, MIN_BQ)
            ro.count_stream_loci(entries.keys, entries.variant, entries.allele, vlo, vhi, b2, m1, n_pos, off,
                                 *fam.loci[smp], K, counts=want[smp])
        ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
    else:
        ks, want = family_counts(orc, entries, fam, K, MIN_BQ, ns)
    return entries, ks, want


def _submit_all(dkb, kc, fam, region):
    for smp in range(kc.n_samples):
        seq, qual, off = fam.reads[smp]
        loci = dkb.ReadLoci(off, *fam.loci[smp]) if region else None
        kc.submit(dkb.pack_reads(seq, qual, off, MIN_BQ), smp, loci=loci)


@pytest.mark.parametrize("region", [False, True])
@pytest.mark.parametrize("sexes", [[M], [M, F]])
def test_sexed_family_end_to_end(dkb, orc, sexes, region):
    fam = synth.make_sexed_family_host(sexes, K, seed=21, err_rate=0.0)
    entries, ks, want = _fam_oracle(dkb, orc, fam, region)
    nv, nc = len(fam.variants), len(sexes)
    wres = io.family_results(orc, ks, want, nv, nc, THR, fam.classes, fam.sexes)
    with dkb.KmerCounter(K, n_children=nc) as kc:
        kc.build_table(entries)
        if region:
            kc.set_regions(*ro.windows(fam.variants, 400))
        _submit_all(dkb, kc, fam, region)
        got = kc.entry_counts().copy()
        kc.set_locus_classes(fam.classes)
        kc.set_child_sexes(fam.sexes)
        res = tuple(x.copy() for x in kc.finalise(THR))
        kc.clear_locus_classes()
        kc.set_child_sexes(None)
        cleared = kc.finalise(THR)[3].copy()
    with dkb.KmerCounter(K, n_children=nc) as kc:  # a fresh context on the same counters
        kc.build_table(entries)
        if region:
            kc.set_regions(*ro.windows(fam.variants, 400))
        _submit_all(dkb, kc, fam, region)
        fresh = kc.finalise(THR)[3].copy()
    assert np.array_equal(got.astype(np.uint64), want) and want.sum() > 0
    hits, dist, nk, calls = res
    calls = calls.reshape(nv, nc)
    assert np.array_equal(hits.astype(np.uint64), wres[0]) and np.array_equal(dist.astype(np.uint64), wres[1])
    assert np.array_equal(nk, wres[2]) and np.array_equal(calls, wres[3])
    assert np.array_equal(cleared, fresh)
    assert np.array_equal(fresh.reshape(nv, nc), io.family_results(orc, ks, want, nv, nc, THR)[3])
    # the designed flips: the son's Y de novo and his X de novo over a carrier father are called
    scen = np.array(fam.scenarios)
    for name in ("y_denovo", "x_denovo_carrier_father"):
        assert (calls[scen == name, 0] == dkb.CALL_DENOVO).all(), name
        assert not (fresh.reshape(nv, nc)[scen == name, 0] & 1).any(), name
    if nc == 2:
        assert (calls[scen == "y_denovo", 1] & dkb.CALL_NO_COPY).all()
    for v, name in enumerate(fam.scenarios):
        _, son, daughter = synth.SEXED_SCENARIOS[name]
        assert calls[v].tolist() == [son if s == M else daughter for s in sexes], name


def test_pipelined_trios_keep_their_settings(dkb, orc):
    """Three independent trios through one context with reduce_push / reduce_flush: the child is
    set male, female, then unknown before each trio's submits, and the classes change before
    the third push.  Each batch's calls follow what was in force at its own push."""
    trios = [synth.make_sexed_family_host([M], K, seed=31, err_rate=0.0),
             synth.make_sexed_family_host([F], K, seed=31, err_rate=0.0),
             synth.make_sexed_family_host([M], K, seed=31, depth=12, err_rate=0.0)]
    entries = dkb.variant_kmers(trios[0].variant_tuples(), K)
    assert all(t.variant_tuples() == trios[0].variant_tuples() for t in trios)
    cls1 = trios[0].classes
    cls2 = np.where(cls1 == A, MT, A).astype(np.uint8)
    settings = [(cls1, M), (cls1, F), (cls2, U)]
    want = []
    for i, (t, (cls, sex)) in enumerate(zip(trios, settings)):
        ks, counts = family_counts(orc, entries, t, K, MIN_BQ, 3)
        want.append((counts, io.family_results(orc, ks, counts, len(t.variants), 1, THR, cls, [sex])))
        # what a batch would get from the settings of the next push: different calls
        nxt = settings[i + 1] if i < 2 else (cls1, M)
        assert not np.array_equal(want[-1][1][3], io.family_results(orc, ks, counts, len(t.variants), 1, THR,
                                                                      nxt[0], [nxt[1]])[3]), i
    got = []
    with dkb.KmerCounter(K) as kc:
        kc.build_table(entries)
        kc.set_locus_classes(cls1)
        for i, (t, (_, sex)) in enumerate(zip(trios, settings)):
            kc.reset_counts()
            kc.set_child_sexes([sex])
            _submit_all(dkb, kc, t, False)
            if i == 2:
                kc.set_locus_classes(cls2)
            kc.reduce_push(THR)
            if i:
                got.append((kc.reduced_counts().copy(),) + tuple(x.copy() for x in kc.results()))
        kc.set_child_sexes([M])  # after the last push: changes nothing of it
        kc.set_locus_classes(cls1)
        kc.reduce_flush(THR)
        got.append((kc.reduced_counts().copy(),) + tuple(x.copy() for x in kc.results()))
    for (counts, wres), g in zip(want, got):
        assert np.array_equal(g[0].astype(np.uint64), counts)
        assert np.array_equal(g[1].astype(np.uint64), wres[0]) and np.array_equal(g[3], wres[2])
        assert np.array_equal(g[4], wres[3][:, 0])
    assert len({g[4].tobytes() for g in got}) == 3


def test_refusals_and_resets(dkb, orc):
    from denovo_kmer_b200 import _lib
    fam = synth.make_sexed_family_host([M], K, seed=41, err_rate=0.0)
    entries = dkb.variant_kmers(fam.variant_tuples(), K)
    nv = len(fam.variants)
    u8 = lambda a: np.ascontiguousarray(a, dtype=np.uint8).ctypes.data_as(_lib.u8p)  # noqa: E731
    with dkb.KmerCounter(K, n_children=2) as kc:
        L, h = kc._L, kc._h
        assert L.dkb_table_set_locus_classes(h, u8(np.zeros(nv)), nv) == _lib.ESTATE  # before the table
        assert L.dkb_table_set_locus_classes(h, None, 0) == _lib.ESTATE
        assert L.dkb_ctx_set_child_sexes(h, u8([M, F]), 2) == _lib.OK  # sexes: any time
        assert L.dkb_ctx_set_child_sexes(h, u8([M]), 1) == _lib.EINVAL
        assert L.dkb_ctx_set_child_sexes(h, u8([M, F, M]), 3) == _lib.EINVAL
        assert L.dkb_ctx_set_child_sexes(h, u8([M, 3]), 2) == _lib.EINVAL
        assert L.dkb_ctx_set_child_sexes(h, None, 2) == _lib.OK and L.dkb_ctx_set_child_sexes(h, None, 0) == _lib.OK
        assert L.dkb_ctx_set_child_sexes(h, None, 1) == _lib.EINVAL
        kc.build_table(entries)
        assert L.dkb_table_set_locus_classes(h, u8(np.zeros(nv + 1)), nv + 1) == _lib.EINVAL
        assert L.dkb_table_set_locus_classes(h, u8(np.zeros(nv - 1)), nv - 1) == _lib.EINVAL
        bad = fam.classes.copy()
        bad[-1] = 4
        assert L.dkb_table_set_locus_classes(h, u8(bad), nv) == _lib.EINVAL
        assert L.dkb_table_set_locus_classes(h, None, nv) == _lib.EINVAL
        with pytest.raises(dkb.DkbError) as ei:
            kc.set_child_sexes([M])
        assert ei.value.code == _lib.EINVAL
    # a new table build resets the classes, not the sexes
    ks, counts = family_counts(orc, entries, fam, K, MIN_BQ, 3)
    with_cls = io.family_results(orc, ks, counts, nv, 1, THR, fam.classes, [M])[3][:, 0]
    male_only = io.family_results(orc, ks, counts, nv, 1, THR, None, [M])[3][:, 0]
    assert not np.array_equal(with_cls, male_only)
    with dkb.KmerCounter(K) as kc:
        kc.set_child_sexes([M])
        kc.build_table(entries)
        kc.set_locus_classes(fam.classes)
        kc.build_table(entries)
        _submit_all(dkb, kc, fam, False)
        assert np.array_equal(kc.finalise(THR)[3], male_only)
        kc.set_locus_classes(fam.classes)  # the son's sex is still set: his Y de novo is called
        assert np.array_equal(kc.finalise(THR)[3], with_cls)

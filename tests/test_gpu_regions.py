"""-m gpu: region-scoped counting (DESIGN.md §2) on the B200 against the region oracle
(tests/region_oracle.c), bit for bit, over the tunings, k, indels, batching, every submit form
and the edges of the read-locus index; the paralog known answer; configs[1] at full size;
and every refusal of the ABI's region calls."""
import numpy as np
import pytest

import region_oracle as ro
from denovo_kmer_b200 import synth

pytestmark = pytest.mark.gpu

THR = (3, 2, 0, 1)
BAM_CODES = {c: i for i, c in enumerate(b"=ACMGRSVTWYHKDBN")}


def _oracle(orc, entries, trio, k, vlo, vhi, min_bq):
    want = np.zeros((3, len(entries)), dtype=np.uint64)
    for smp in range(3):
        seq, qual, off = trio.reads[smp]
        b2, m1, n_pos = orc.pack_stream(seq, qual, off, min_bq)
        lo, hi = trio.loci[smp]
        ro.count_stream_loci(entries.keys, entries.variant, entries.allele, vlo, vhi, b2, m1, n_pos, off, lo, hi, k,
                             counts=want[smp])
    return want


def _gpu(dkb, entries, trio, k, vlo, vhi, min_bq, tuning=None, hints=True, batches=1, form="submit"):
    with dkb.KmerCounter(k, tuning=tuning) as kc:
        kc.build_table(entries, use_window_hints=hints)
        if vlo is not None:
            kc.set_regions(vlo, vhi)
        for smp in range(3):
            seq, qual, off = trio.reads[smp]
            lo, hi = trio.loci[smp]
            cuts = np.linspace(0, len(off) - 1, batches + 1).astype(int)
            for a, b in zip(cuts[:-1], cuts[1:]):
                if b == a:
                    continue
                boff = off[a:b + 1]
                loci = None if vlo is None else dkb.ReadLoci(boff, lo[a:b], hi[a:b])
                _submit(dkb, kc, form, seq, qual, boff, smp, min_bq, loci)
        got = kc.entry_counts().copy()
        res = kc.finalise(THR)
        tun = kc.tuning()
    return got, res, tun


def _four_bit(seq, off):
    """ASCII reads -> BAM 4-bit codes, every read on a byte boundary, reads back to back."""
    out = []
    for r in range(len(off) - 1):
        s = seq[int(off[r]):int(off[r + 1])].tobytes()
        codes = [BAM_CODES.get(c, 15) for c in s.upper()] + ([0] if len(s) % 2 else [])
        out += [codes[i] << 4 | codes[i + 1] for i in range(0, len(codes), 2)]
    return np.array(out, dtype=np.uint8)


def _submit(dkb, kc, form, seq, qual, off, smp, min_bq, loci):
    import torch
    a, b = int(off[0]), int(off[-1])
    if form == "reads":  # offsets[0] != 0 is kept: the library reads seq/qual from offsets[0]
        kc.submit_reads(seq, qual, off, smp, min_bq, loci=loci)
        return
    if form == "reads4":
        rel = off - off[0]
        kc.submit_reads(_four_bit(seq[a:b], rel), qual[a:b], rel, smp, min_bq, four_bit=True,
                        loci=None if loci is None else dkb.ReadLoci(rel, loci.lo, loci.hi))
        return
    st = dkb.pack_reads(seq[a:b], qual[a:b], off - off[0], min_bq)
    if form == "submit":
        kc.submit(st, smp, loci=loci)
    elif form == "sparse":
        zoff, zbytes = dkb.mask_to_zero_list(st.mask1, st.n_positions)
        kc.submit_sparse(st.bases2, zoff, zbytes, st.n_positions, smp, loci=loci)
    elif form == "device":
        b2 = torch.from_numpy(st.bases2.view(np.int32).copy()).cuda()
        m1 = torch.from_numpy(st.mask1.view(np.int32).copy()).cuda()
        kc.submit_device(b2.data_ptr(), m1.data_ptr(), st.n_positions, smp, loci=loci)
        kc.sync()  # the tensors go out of scope here


def _check(dkb, orc, trio, k, pad=500, min_bq=20, drop_shared=True, **kw):
    entries = dkb.variant_kmers(trio.variant_tuples(), k, drop_shared=drop_shared)
    vlo, vhi = ro.windows(trio.variants, pad)
    want = _oracle(orc, entries, trio, k, vlo, vhi, min_bq)
    got, res, tun = _gpu(dkb, entries, trio, k, vlo, vhi, min_bq, **kw)
    bad = np.nonzero(got.astype(np.uint64) != want)
    assert len(bad[0]) == 0, (tun, len(bad[0]), [(int(s), int(e), int(got[s, e]), int(want[s, e])) for s, e in zip(*bad)][:5])
    assert want.sum() > 0
    return entries, want, res


def _trimmed(trio, frac=0.5, seed=0):
    """Windows that cut some reads out: the trio with half its reads moved to far-away loci."""
    rng = np.random.default_rng(seed)
    for smp in range(3):
        lo, hi = trio.loci[smp]
        far = rng.random(len(lo)) < frac
        lo[far] += np.uint64(1 << 30)
        hi[far] += np.uint64(1 << 30)
    return trio


TUNINGS = [None, (15, 1, 1), (15, 1, 2), (13, 1, 2), (15, 2, 1), (15, 2, 2), (14, 4, 1), (14, 4, 2), (12, 1, 1),
           (9, 2, 1), (15, 8, 2), (13, 8, 1), (15, 16, 2), (9, 16, 1), (15, 16, 2, 2), (14, 4, 1, 2), (15, 2, 2, 2),
           (13, 8, 2, 2)]


@pytest.mark.parametrize("tuning", TUNINGS)
@pytest.mark.parametrize("hints", [True, False])
def test_region_parity_tunings(dkb, orc, tuning, hints):
    trio = _trimmed(synth.make_trio_host(200_000, 12, 40, 31, seed=5))
    _check(dkb, orc, trio, 31, pad=300, tuning=tuning, hints=hints)


@pytest.mark.parametrize("gate", ["0", "1"])
@pytest.mark.parametrize("tuning", [(15, 16, 2, 2), (13, 8, 1, 2), (9, 16, 2, 2)])
def test_region_parity_gated_lookups(dkb, orc, tuning, gate, monkeypatch):
    monkeypatch.setenv("DKB_GATE", gate)
    trio = _trimmed(synth.make_trio_host(150_000, 14, 30, 31, seed=77, n_rate=0.01, lowq_frac=0.08, ragged=True))
    _check(dkb, orc, trio, 31, tuning=tuning)


@pytest.mark.parametrize("k", [15, 21, 31])
def test_region_parity_k(dkb, orc, k):
    trio = _trimmed(synth.make_trio_host(100_000, 10, 20, k, seed=7 + k))
    _check(dkb, orc, trio, k, pad=100)
    _check(dkb, orc, trio, k, pad=100, hints=False, tuning=(0, 2, 0))


@pytest.mark.parametrize("drop_shared", [True, False])
def test_region_parity_indels(dkb, orc, drop_shared):
    trio = _trimmed(synth.make_trio_host(150_000, 15, 40, 31, seed=11, indel_frac=0.6))
    _check(dkb, orc, trio, 31, pad=50, drop_shared=drop_shared)


def test_region_parity_ragged_batches(dkb, orc):
    trio = _trimmed(synth.make_trio_host(100_000, 15, 20, 21, seed=13, ragged=True, n_rate=0.01, lowq_frac=0.1))
    _check(dkb, orc, trio, 21, batches=7)


def test_region_results_equal_per_variant_fetch(dkb, orc):
    """dkb_finalise's per-variant statistics and calls in region mode equal those of the plain
    per-variant read fetch (no stream walk involved)."""
    k = 31
    trio = _trimmed(synth.make_trio_host(20_000, 12, 8, k, seed=31, indel_frac=0.3), frac=0.3, seed=2)
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    vlo, vhi = ro.windows(trio.variants, 200)
    want = ro.py_fetch_counts(entries.keys, entries.variant, entries.allele, len(trio.variants), vlo, vhi,
                              [ro.trio_reads(trio, s) for s in range(3)], k, 20)
    got, (hits, dist, nk, calls), _ = _gpu(dkb, entries, trio, k, vlo, vhi, 20, batches=3)
    assert np.array_equal(got.astype(np.uint64), want) and want.sum() > 0
    ks = orc.KmerSet(entries.keys, entries.variant, entries.allele)
    o_hits, o_dist, o_nk = ks.variant_stats(want, len(trio.variants))
    assert np.array_equal(hits.astype(np.uint64), o_hits) and np.array_equal(dist.astype(np.uint64), o_dist)
    assert np.array_equal(nk, o_nk) and np.array_equal(calls, orc.calls(o_hits, o_dist, THR))


def test_region_reduces_to_whole_stream(dkb, orc):
    k = 31
    trio = synth.make_trio_host(100_000, 12, 20, k, seed=3, indel_frac=0.3)
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    nv = len(trio.variants)
    whole, _, _ = _gpu(dkb, entries, trio, k, None, None, 20)
    from helpers import oracle_counts
    _, want = oracle_counts(orc, entries, trio, k, 20)
    assert np.array_equal(whole.astype(np.uint64), want) and want.sum() > 0
    cover, _, _ = _gpu(dkb, entries, trio, k, np.zeros(nv, np.uint64), np.full(nv, 1 << 40, np.uint64), 20)
    assert np.array_equal(cover, whole)
    miss, _, _ = _gpu(dkb, entries, trio, k, np.full(nv, 1 << 40, np.uint64), np.full(nv, (1 << 40) + 9, np.uint64), 20)
    assert miss.sum() == 0
    with dkb.KmerCounter(k) as kc:  # region mode switched off again
        kc.build_table(entries)
        kc.set_regions(np.zeros(nv, np.uint64), np.zeros(nv, np.uint64))
        kc.clear_regions()
        for smp in range(3):
            kc.submit(dkb.pack_reads(*trio.reads[smp], 20), smp)
        assert np.array_equal(kc.entry_counts().astype(np.uint64), want)


@pytest.mark.parametrize("form", ["submit", "sparse", "reads", "reads4", "device"])
def test_region_every_submit_form(dkb, orc, form):
    trio = _trimmed(synth.make_trio_host(100_000, 12, 20, 31, seed=19, indel_frac=0.3, ragged=True))
    _check(dkb, orc, trio, 31, pad=200, batches=3, form=form)


def test_region_edges(dkb, orc):
    """Hand-made batch: reads crossing 2048-position tiles, reads longer than a tile (5 000
    bases), empty reads, unmapped reads, an empty variant window, a k-mer ending at the
    stream's last position, a one-read batch, and offsets[0] != 0."""
    k = 31
    rng = np.random.default_rng(4)
    genome = synth.make_genome(60_000, 8)
    variants = synth.plant_variants(genome, 12, k, 9)
    trio = synth.Trio(k, genome, variants)
    alt = synth.apply_variants(genome, variants)
    rp = synth.hap_ref_positions(genome, variants)
    lens = [5000, 0, 150, 3000, 0, 0, 2100, 2048, 31, 4000, 1, 150] * 6
    seqs, lo, hi = [], [], []
    for i, n in enumerate(lens):
        s = int(rng.integers(0, len(alt) - max(n, 1)))
        seqs.append(alt[s:s + n])
        lo.append(int(rp[s]))
        hi.append(int(rp[s + n - 1]) + 1 if n else int(rp[s]))
    # the last read ends on a variant's alt k-mer: a k-mer ends at the stream's last position
    # (before its separator)
    v = variants[-1]
    e = v.pos + 1
    j = int(np.searchsorted(rp, v.pos))
    seqs.append(alt[j - 40:j + 1])
    lo.append(int(rp[j - 40]))
    hi.append(e)
    seq = np.concatenate(seqs)
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(x) for x in seqs])
    qual = np.full(len(seq), 30, dtype=np.uint8)
    lo, hi = np.array(lo, np.uint64), np.array(hi, np.uint64)
    hi[3::9] = lo[3::9]  # unmapped
    trio.reads = {s: (seq, qual, off) for s in range(3)}
    trio.loci = {s: (lo.copy(), hi.copy()) for s in range(3)}
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    vlo, vhi = ro.windows(variants, 2000)
    vhi[2] = vlo[2]  # empty window
    want = _oracle(orc, entries, trio, k, vlo, vhi, 20)
    assert want[:, entries.variant == len(variants) - 1].sum() > 0
    for tuning in [None, (15, 2, 2), (15, 16, 2, 2), (12, 1, 1)]:
        for batches in (1, 5):
            got, _, _ = _gpu(dkb, entries, trio, k, vlo, vhi, 20, tuning=tuning, batches=batches)
            assert np.array_equal(got.astype(np.uint64), want), (tuning, batches)
        # offsets[0] != 0: reads submitted as the tail of the caller's arrays
        got, _, _ = _gpu(dkb, entries, trio, k, vlo, vhi, 20, tuning=tuning, batches=3, form="reads")
        assert np.array_equal(got.astype(np.uint64), want), tuning
    # a one-read batch: the long read alone
    one = synth.Trio(k, genome, variants)
    one.reads = {s: (seq, qual, off[:2]) for s in range(3)}
    one.loci = {s: (lo[:1].copy(), hi[:1].copy()) for s in range(3)}
    got, _, _ = _gpu(dkb, entries, one, k, vlo, vhi, 20)
    assert np.array_equal(got.astype(np.uint64), _oracle(orc, entries, one, k, vlo, vhi, 20))


def test_region_paralog_known_answer(dkb):
    """A de novo candidate whose ALT context also sits at a far-away paralog: whole-stream
    counting sees the alt k-mers in both parents; counting only reads aligned within 500 bases
    calls it de novo again.  No other call byte changes.  (Error-free reads: a sequencing error
    can put a de novo allele's k-mer into a parent's read by chance.)"""
    k = 31
    trio = synth.make_trio_host(200_000, 20, 30, k, seed=12, paralog_frac=0.3, err_rate=0.0)
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    vlo, vhi = ro.windows(trio.variants, 500)
    _, (_, _, _, whole), _ = _gpu(dkb, entries, trio, k, None, None, 20)
    _, (_, _, _, region), _ = _gpu(dkb, entries, trio, k, vlo, vhi, 20)
    par = np.zeros(len(trio.variants), dtype=bool)
    par[trio.paralogs] = True
    both = dkb.CALL_MOTHER_ALT | dkb.CALL_FATHER_ALT
    assert ((whole & both) == both)[par].all(), whole[par]
    assert ((whole & both) == 0)[~par & ~np.array([v.inherited for v in trio.variants])].all()
    assert (region[par] == dkb.CALL_DENOVO).all(), region[par]
    assert np.array_equal(region[~par], whole[~par])


def test_region_config1_full_size(dkb, orc):
    """configs[1] (64 Mb, 30x, 10 000 candidates, k = 31) in region mode with +-500-base windows:
    the bench generator's streams with the loci of its read starts, every counter equal to the
    region oracle on the scanned streams."""
    import torch
    import bench
    a = bench.parse_args([])
    dev = torch.device("cuda:0")
    genome, variants, tuples = bench.make_variants(a, synth)
    entries = dkb.variant_kmers(tuples, a.k)
    lut = np.zeros(256, dtype=np.uint8)
    for i, ch in enumerate(b"ACGT"):
        lut[ch] = i
    mother_var = [v for v in variants if v.inherited]
    haps = [[genome, synth.apply_variants(genome, variants)], [genome, synth.apply_variants(genome, mother_var)],
            [genome, genome]]
    refpos = [[None, synth.hap_ref_positions(genome, variants)], [None, synth.hap_ref_positions(genome, mother_var)],
              [None, None]]
    n_reads = int(len(genome) * a.depth / bench.READ_LEN) // 128 * 128
    vlo, vhi = ro.windows(variants, 500)
    want = np.zeros((3, len(entries)), dtype=np.uint64)
    with dkb.KmerCounter(a.k) as kc:
        kc.build_table(entries)
        kc.set_regions(vlo, vhi)
        for s in range(3):
            hs = [torch.from_numpy(lut[h]).to(dev) for h in haps[s]]
            b2, m1, n_pos, _, meta = synth.make_sample_device(hs, n_reads, bench.READ_LEN, 1000 + s, dev,
                                                              return_meta=True)
            del hs
            off, lo, hi = synth.device_read_loci(meta, refpos[s], bench.READ_LEN)
            kc.submit_device(b2.data_ptr(), m1.data_ptr(), n_pos, s, loci=dkb.ReadLoci(off, lo, hi))
            kc.sync()
            ro.count_stream_loci(entries.keys, entries.variant, entries.allele, vlo, vhi, b2.cpu().numpy(),
                                 m1.cpu().numpy(), n_pos, off, lo, hi, a.k, counts=want[s])
            del b2, m1
            torch.cuda.empty_cache()
        got = kc.entry_counts().copy()
        tun = kc.tuning()
    bad = int((got.astype(np.uint64) != want).sum())
    assert bad == 0, f"{bad} of {want.size} counters differ (tuning {tun})"
    assert want.sum() > 1_000_000


def test_region_refusals(dkb):
    from denovo_kmer_b200 import _lib
    L = _lib.lib()
    import ctypes as C
    import torch
    k = 31
    trio = synth.make_trio_host(20_000, 4, 4, k, seed=2)
    entries = dkb.variant_kmers(trio.variant_tuples(), k)
    nv = len(trio.variants)
    seq, qual, off = trio.reads[0]
    st = dkb.pack_reads(seq, qual, off, 20)
    lo, hi = trio.loci[0]
    u64 = lambda a: np.ascontiguousarray(a, dtype=np.uint64).ctypes.data_as(_lib.u64p)  # noqa: E731
    with dkb.KmerCounter(k) as kc:
        h = kc._h
        z = np.zeros(nv, np.uint64)
        assert L.dkb_table_set_regions(h, u64(z), u64(z), nv) == _lib.ESTATE  # before the table
        kc.build_table(entries)
        assert L.dkb_batch_set_loci(h, u64(off), u64(lo), u64(hi), len(off) - 1) == _lib.ESTATE  # whole-stream
        assert L.dkb_table_set_regions(h, u64(z), u64(z), nv + 1) == _lib.EINVAL
        assert L.dkb_table_set_regions(h, u64(z), None, nv) == _lib.EINVAL
        kc.set_regions(*ro.windows(trio.variants, 100))
        # a submit without loci
        assert L.dkb_batch_submit(h, st.bases2.ctypes.data, st.mask1.ctypes.data, st.n_positions, 0) == _lib.ESTATE
        # loci of a different batch
        assert L.dkb_batch_set_loci(h, u64(off[:-1]), u64(lo[:-1]), u64(hi[:-1]), len(off) - 2) == _lib.OK
        assert L.dkb_batch_submit(h, st.bases2.ctypes.data, st.mask1.ctypes.data, st.n_positions, 0) == _lib.EINVAL
        bad = off.copy()
        bad[3] = bad[4] + 1
        assert L.dkb_batch_set_loci(h, u64(bad), u64(lo), u64(hi), len(off) - 1) == _lib.EINVAL  # descending
        assert L.dkb_batch_set_loci(h, u64(off), u64(lo), u64(hi), C.c_size_t(1 << 32)) == _lib.EINVAL
        b2 = torch.from_numpy(st.bases2.view(np.int32).copy()).cuda()
        m1 = torch.from_numpy(st.mask1.view(np.int32).copy()).cuda()
        n = (C.c_uint64 * 1)(st.n_positions)
        assert L.dkb_batch_submit_device_multi(h, 1, (C.c_void_p * 1)(b2.data_ptr()), (C.c_void_p * 1)(m1.data_ptr()),
                                               n, (C.c_int * 1)(0)) == _lib.ESTATE
        # every single-batch form: a submit refused for a bad sample uses up its loci, and without
        # loci a bad sample is refused for the missing loci
        for form in ("submit", "sparse", "reads", "reads4", "device"):
            for smp, loci, code in ((3, dkb.ReadLoci(off, lo, hi), _lib.EINVAL), (0, None, _lib.ESTATE),
                                    (3, None, _lib.ESTATE)):
                with pytest.raises(dkb.DkbError) as ei:
                    _submit(dkb, kc, form, seq, qual, off, smp, 20, loci)
                assert ei.value.code == code, (form, smp, loci is not None)
        kc.profile_counters(True)  # region mode has no profiling kernels: refused, never ungated
        assert L.dkb_batch_set_loci(h, u64(off), u64(lo), u64(hi), len(off) - 1) == _lib.OK
        assert L.dkb_batch_submit(h, st.bases2.ctypes.data, st.mask1.ctypes.data, st.n_positions, 0) == _lib.ESTATE
        kc.profile_counters(False)
        kc.submit(st, 0, loci=dkb.ReadLoci(off, lo, hi))  # and a proper one still works
        kc.sync()
        assert kc.entry_counts().sum() > 0
        # a new table returns to whole-stream counting: loci are refused again
        kc.build_table(entries)
        assert L.dkb_batch_set_loci(h, u64(off), u64(lo), u64(hi), len(off) - 1) == _lib.ESTATE
